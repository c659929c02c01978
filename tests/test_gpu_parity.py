"""GPU: the CUDA path through the C ABI against the CPU oracle, the goldens and the oracle KATs.

Bars (BASELINE.json north_star): hit step, device id, missile cost bit-exact; min distance within
1e-6 relative (MIN_DIST_RTOL below).  Stronger checks where the arithmetic allows: the STRICT kernel
is bit-identical to the oracle's sqrt3 mode on the full state."""
import json
import os
import subprocess

import numpy as np
import pytest
from conftest import ROOT, CASES, GOLDEN, case_path, golden_lines

pytestmark = pytest.mark.gpu
MIN_DIST_RTOL = 1e-6  # tolerance the north star states for output line 1


def ulps(a, b):
    return np.abs(a - b) / np.spacing(np.maximum(np.abs(a), np.abs(b)))


@pytest.fixture(scope="module")
def kats():
    return json.load(open(os.path.join(GOLDEN, "oracle_kats.json")))


# ---- state-level parity --------------------------------------------------------------------------
@pytest.mark.parametrize("case,steps", [("b20", 3000), ("b100", 1000), ("b200", 400), ("b512", 60), ("b1024", 20)])
def test_strict_kernel_state_is_bit_identical_to_oracle(nb, oracle, case, steps):
    s = nb.read_input(case_path(case))
    q, v = s.q.copy(), s.v.copy()
    nb.run_steps(0, steps, s.n, q, v, s.m, s.is_device, math=nb.MATH_STRICT)
    qo, vo = s.q.copy(), s.v.copy()
    oracle.run_steps(oracle.MODE_SQRT3, s.n, qo, vo, s.m, s.is_device, 0, steps)
    assert np.array_equal(q, qo)
    assert np.array_equal(v, vo)


@pytest.mark.parametrize("case,steps", [("b20", 3000), ("b60", 1000), ("b100", 1000), ("b200", 400), ("b512", 60),
                                        ("b1024", 20)])
def test_fast_kernel_state_matches_oracle(nb, oracle, case, steps):
    """Fast math (rsqrt seed + correction, FMA, lane-split sums): positions equal to the last bit or
    two, velocities to 1e-12 relative — SURVEY App. B explains why the rounded state absorbs it."""
    s = nb.read_input(case_path(case))
    q, v = s.q.copy(), s.v.copy()
    nb.run_steps(0, steps, s.n, q, v, s.m, s.is_device, math=nb.MATH_FAST)
    qo, vo = s.q.copy(), s.v.copy()
    oracle.run_steps(oracle.MODE_STRICT, s.n, qo, vo, s.m, s.is_device, 0, steps)
    assert ulps(q, qo).max() <= 2
    assert np.allclose(v, vo, rtol=1e-12, atol=0)


def test_run_step_is_the_reference_operator(nb, oracle):
    """run_step(step, ...) one step at a time == many steps in one call (step index drives the device mass)."""
    s = nb.read_input(case_path("b30"))
    q, v = s.q.copy(), s.v.copy()
    for step in range(1, 6):
        nb.run_step(step, s.n, q, v, s.m, s.is_device, math=nb.MATH_STRICT)
    q2, v2 = s.q.copy(), s.v.copy()
    nb.run_steps(0, 5, s.n, q2, v2, s.m, s.is_device, math=nb.MATH_STRICT)
    assert np.array_equal(q, q2) and np.array_equal(v, v2)
    qo, vo = s.q.copy(), s.v.copy()
    oracle.run_steps(oracle.MODE_SQRT3, s.n, qo, vo, s.m, s.is_device, 0, 5)
    assert np.array_equal(q, qo) and np.array_equal(v, vo)
    # a later step index gives a different device mass, hence a different state
    q3, v3 = s.q.copy(), s.v.copy()
    nb.run_steps(100, 105, s.n, q3, v3, s.m, s.is_device, math=nb.MATH_STRICT)
    assert not np.array_equal(v3, v2)
    qo, vo = s.q.copy(), s.v.copy()
    oracle.run_steps(oracle.MODE_SQRT3, s.n, qo, vo, s.m, s.is_device, 100, 105)
    assert np.array_equal(q3, qo) and np.array_equal(v3, vo)


@pytest.mark.parametrize("n", [1, 2, 3, 31, 33, 1000, 1024])
def test_edge_sizes_small_path(nb, oracle, n):
    """Ragged / minimal systems through the persistent kernel (n == 1 has no pair at all)."""
    s = nb.synthetic_system(max(n, 6), seed=n)
    q, v, m, dev = (s.q.reshape(3, -1)[:, :n].copy().reshape(-1), s.v.reshape(3, -1)[:, :n].copy().reshape(-1),
                    s.m[:n].copy(), s.is_device[:n].copy())
    if n >= 3:
        dev[-1] = 1
    qo, vo = q.copy(), v.copy()
    nb.run_steps(0, 7, n, q, v, m, dev, math=nb.MATH_STRICT)
    oracle.run_steps(oracle.MODE_SQRT3, n, qo, vo, m, dev, 0, 7)
    assert np.array_equal(q, qo) and np.array_equal(v, vo)


# ---- the three queries against the goldens ---------------------------------------------------------
@pytest.mark.parametrize("case", CASES)
def test_solve_matches_golden(nb, case, kats):
    s = nb.read_input(case_path(case))
    g = golden_lines(case)
    ans = nb.solve(s, gpus=[0], all_devices=True)  # INDEPENDENT plan: every device's trajectory from step 0
    assert ans.hit_time_step == g["hit_time_step"]            # bit-exact
    assert ans.gravity_device_id == g["gravity_device_id"]    # bit-exact
    assert ans.missile_cost == g["missile_cost"]              # bit-exact
    assert abs(ans.min_dist - g["min_dist"]) <= MIN_DIST_RTOL * g["min_dist"]
    if case in kats:  # intermediate known answers of the oracle
        k = kats[case]
        assert ans.argmin_step == k["argmin_step"]
        for j, d in enumerate(k["devices"]):
            assert ans.device_index[j] == d["index"]
            assert ans.reach_step[j] == d["reach_step"]
            assert ans.q3_hit_step[j] == d["q3_hit_step"]


@pytest.mark.parametrize("case", CASES)
def test_solve_chain_plan_matches_golden(nb, case, kats):
    """Default plan on one GPU (fewer GPUs than trajectories): query 3 forked from query 2 at most one chunk before the
    missile arrives, candidates in order of cost, search stopped at the first saviour (hw5.cu:438-530, 575-588).  Same
    answers as the goldens; the devices it did simulate agree with the oracle's KATs, the others read -3."""
    s = nb.read_input(case_path(case))
    g = golden_lines(case)
    ans = nb.solve(s, gpus=[0])
    assert (ans.hit_time_step, ans.gravity_device_id, ans.missile_cost) == (g["hit_time_step"], g["gravity_device_id"], g["missile_cost"])
    assert abs(ans.min_dist - g["min_dist"]) <= MIN_DIST_RTOL * g["min_dist"]
    if case in kats:
        k = kats[case]
        assert ans.argmin_step == k["argmin_step"]
        simulated = 0
        for j, d in enumerate(k["devices"]):
            assert ans.reach_step[j] == d["reach_step"]
            if ans.q3_hit_step[j] != -3:
                simulated += 1
                assert ans.q3_hit_step[j] == d["q3_hit_step"]
        saviours = [d for d in k["devices"] if d["q3_hit_step"] == -2]
        assert simulated == (1 if saviours else len(k["devices"]))  # the cheapest saviour is the first candidate tried


def test_solve_output_file_is_byte_identical_for_small_goldens(nb, tmp_path):
    """Stronger than the bar: on these inputs even line 1 comes out to the last digit."""
    for case in ("b20", "b30", "b50"):
        out = tmp_path / (case + ".out")
        nb.hw5_main(case_path(case), str(out), 1)
        assert out.read_text() == golden_lines(case)["text"]


def test_hw5_cli_binary(nb, tmp_path):
    out = tmp_path / "b40.out"
    r = subprocess.run([nb.HW5_PATH, case_path("b40"), str(out)], capture_output=True)
    assert r.returncode == 0, r.stderr
    g = golden_lines("b40")
    a, b, c = out.read_text().split("\n")[:3]
    assert b == str(g["hit_time_step"]) and c == g["text"].split("\n")[2]
    assert abs(float(a) - g["min_dist"]) <= MIN_DIST_RTOL * g["min_dist"]


def test_solve_strict_math_matches_golden_b20(nb):
    s = nb.read_input(case_path("b20"))
    g = golden_lines("b20")
    ans = nb.solve(s, gpus=[0], math=nb.MATH_STRICT)
    assert nb.format_output(ans.min_dist, ans.hit_time_step, ans.gravity_device_id, ans.missile_cost) == g["text"]


def test_no_hit_defaults(nb, oracle):
    """No collision inside the horizon: -2 and '-1 0' (hw5.cu:545-548,568); no golden pins this path."""
    s = nb.read_input(case_path("b20"))
    ans = nb.solve(s, gpus=[0], n_steps=1000)
    ref = oracle.solve(oracle.MODE_STRICT, s, n_steps=1000)
    assert (ans.hit_time_step, ans.gravity_device_id, ans.missile_cost) == (-2, -1, 0.0)
    assert ans.min_dist == ref.min_dist and ans.argmin_step == ref.argmin_step


# ---- trajectories / events -------------------------------------------------------------------------
def test_solve_plans_on_edge_cases(nb, oracle):
    """Both scheduler plans against the oracle where the goldens have no case: zero steps, one step, no devices at all,
    a collision in the initial state (nbody.cc:131-137 tests step 0 too), fewer steps than any missile needs."""
    base = nb.read_input(case_path("b20"))
    nodev = base.copy()
    nodev.is_device[:] = 0
    crash = base.copy()
    for k in range(3):
        crash.q[k * crash.n + crash.asteroid] = crash.q[k * crash.n + crash.planet] + 1.0e6
    big = nb.read_input(case_path("b200"))  # n >= 128: the whole-GPU kernel
    bigcrash = big.copy()
    for k in range(3):
        bigcrash.q[k * big.n + big.asteroid] = bigcrash.q[k * big.n + big.planet] + 1.0e6
    for name, s, n_steps in (("zero steps", base, 0), ("one step", base, 1), ("no devices", nodev, 3000),
                             ("hit at step 0", crash, 50), ("short", base, 2500), ("zero steps, b200", big, 0),
                             ("hit at step 0, b200", bigcrash, 40), ("short, b200", big, 300)):
        ref = oracle.solve(oracle.MODE_STRICT, s, n_steps=n_steps)
        for all_devices in (False, True):
            ans = nb.solve(s, gpus=[0], n_steps=n_steps, all_devices=all_devices)
            assert (ans.hit_time_step, ans.gravity_device_id, ans.missile_cost) == (
                ref.hit_time_step, ref.gravity_device_id, ref.missile_cost), (name, all_devices)
            assert abs(ans.min_dist - ref.min_dist) <= MIN_DIST_RTOL * ref.min_dist, (name, all_devices)


def test_trajectory_events_match_oracle(nb, oracle):
    s = nb.read_input(case_path("b30"))
    for kind, okind, dd in ((nb.KIND_Q1, oracle.KIND_Q1, -1), (nb.KIND_Q2, oracle.KIND_Q2, -1),
                            (nb.KIND_Q3, oracle.KIND_Q3, 28), (nb.KIND_Q3, oracle.KIND_Q3, 29)):
        t = nb.Trajectory(s, kind, dd)
        ev = t.run(nb.N_STEPS)
        oev, qo, vo = oracle.trajectory(oracle.MODE_STRICT, okind, s, dd)
        assert ev.hit_step == oev.hit_step and ev.destroyed_step == oev.destroyed_step
        assert ev.argmin_step == oev.argmin_step and ev.steps_done == oev.steps_done
        assert ev.cost == oev.cost
        assert abs(ev.min_d2 - oev.min_d2) <= 2e-6 * oev.min_d2
        assert list(ev.reach_step[:ev.n_reach]) == list(oev.reach_step[:oev.n_reach])
        q, v, m, step = t.state()
        assert step == oev.steps_done
        assert ulps(q, qo).max() <= 4
        if kind == nb.KIND_Q3:
            assert m[dd] == 0.0  # hw5.cu:306
        t.close()


@pytest.mark.parametrize("n_dev", [33, 40, 64])
def test_grid_kernel_more_than_32_devices(nb, oracle, n_dev):
    """The grid kernel's observer warp keeps two gravity devices per lane (NB_MAX_DEVICES = 64; hw5.cu:265-309 loops over
    the devices on one thread).  b200 with n_dev of its bodies declared devices: query 2 (every device's missile-reach step)
    and a query-3 trajectory of a device of the second half of the list against the oracle, 30 000 steps."""
    import copy
    s = copy.copy(nb.read_input(case_path("b200")))
    dev = np.zeros(s.n, dtype=np.uint8)
    ids = [i for i in range(s.n) if i not in (s.planet, s.asteroid)][-n_dev:]
    dev[ids] = 1
    s.is_device = dev
    steps = 30000
    for kind, okind, dd in ((nb.KIND_Q2, oracle.KIND_Q2, -1), (nb.KIND_Q3, oracle.KIND_Q3, 197), (nb.KIND_Q3, oracle.KIND_Q3, ids[32])):
        t = nb.Trajectory(s, kind, dd)
        ev = t.run(steps)
        oev, qo, vo = oracle.trajectory(oracle.MODE_SQRT3, okind, s, dd, n_steps=steps)
        assert ev.n_reach == oev.n_reach == n_dev
        assert list(ev.reach_step[:n_dev]) == list(oev.reach_step[:n_dev])
        assert (ev.hit_step, ev.destroyed_step, ev.argmin_step, ev.steps_done, ev.cost) == \
               (oev.hit_step, oev.destroyed_step, oev.argmin_step, oev.steps_done, oev.cost)
        assert abs(ev.min_d2 - oev.min_d2) <= 2e-6 * oev.min_d2
        q, v, m, step = t.state()
        assert ulps(q, qo).max() <= 4
        if kind == nb.KIND_Q3 and ev.destroyed_step != -2:
            assert m[dd] == 0.0
        t.close()


def test_trajectory_resume_and_fork(nb):
    """Stopping and resuming a persistent trajectory changes nothing; a fork at the missile-reach
    step (hw5.cu:275-284 snapshot -> :482-483 restore) equals the trajectory simulated from step 0."""
    s = nb.read_input(case_path("b50"))
    a = nb.Trajectory(s, nb.KIND_Q2)
    ea = a.run(nb.N_STEPS)
    b = nb.Trajectory(s, nb.KIND_Q2)
    for end in (1, 2, 1000, 87218, 87219, nb.N_STEPS):
        eb = b.run(end)
    assert eb.as_dict() == ea.as_dict()
    assert all(np.array_equal(x, y) for x, y in zip(a.state()[:2], b.state()[:2]))
    r = ea.reach_step[0]  # device 48
    c = nb.Trajectory(s, nb.KIND_Q2)
    c.run(r)
    f = c.fork(nb.KIND_Q3, 48)
    ef = f.run(nb.N_STEPS)
    d = nb.Trajectory(s, nb.KIND_Q3, 48)
    ed = d.run(nb.N_STEPS)
    assert (ef.hit_step, ef.destroyed_step, ef.cost) == (ed.hit_step, ed.destroyed_step, ed.cost) == (-2, r, 5.23324e9)
    assert all(np.array_equal(x, y) for x, y in zip(f.state()[:2], d.state()[:2]))
    for t in (a, b, c, d, f):
        t.close()


def test_error_codes_on_gpu(nb):
    s = nb.read_input(case_path("b20"))
    with pytest.raises(nb.NbodyError) as e:
        nb.Trajectory(s, nb.KIND_Q1, gpu=99)
    assert e.value.code == nb.NB_ERR_NO_GPU
    big = nb.synthetic_system(2048)
    with pytest.raises(nb.NbodyError) as e:
        nb.Trajectory(big, nb.KIND_Q1)
    assert e.value.code == nb.NB_ERR_UNSUPPORTED
    with pytest.raises(nb.NbodyError) as e:
        nb.Trajectory(s, nb.KIND_Q3, destroy_device=500)
    assert e.value.code == nb.NB_ERR_ARG


def test_grid_kernel_forced_on_small_systems(nb, tmp_path):
    """The whole-GPU cooperative kernel is normally used from n = 256 up; force it on b100 / b200
    (13 / 25 blocks, ragged last block) in a subprocess and compare with the goldens and the KATs."""
    import sys
    code = (
        "import importlib, json, sys\n"
        "sys.path.insert(0, %r)\n"
        "nb = importlib.import_module('nthu_ipc_nbody-simulation_b200')\n"
        "out = {}\n"
        "for case in ('b100', 'b200', 'b90'):\n"
        "    s = nb.read_input(%r + '/' + case + '.in')\n"
        "    a = nb.solve(s, gpus=[0], all_devices=True)\n"
        "    out[case] = dict(text=nb.format_output(a.min_dist, a.hit_time_step, a.gravity_device_id, a.missile_cost),\n"
        "                     argmin=a.argmin_step, reach=list(a.reach_step[:a.n_devices]), q3=list(a.q3_hit_step[:a.n_devices]))\n"
        "print(json.dumps(out))\n") % (os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                                        os.path.join(GOLDEN, "testcases"))
    env = dict(os.environ, NB_GRID_MIN_N="16")
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, env=env, timeout=600)
    assert r.returncode == 0, r.stderr.decode()[-2000:]
    out = json.loads(r.stdout.decode().strip().split("\n")[-1])
    # the exchange knobs change timing only, never results: no multicast / clusters of 2, copies issued far too early
    # (every record stale at first: all of them go through the poll-and-patch path) and one system per launch
    for knobs in (dict(NB_GRID_CS="1"), dict(NB_GRID_CS="2", NB_GRID_DELAY="0", NB_GRID_T="1")):
        r2 = subprocess.run([sys.executable, "-c", code.replace("('b100', 'b200', 'b90')", "('b200',)")], capture_output=True,
                            env=dict(env, **knobs), timeout=600)
        assert r2.returncode == 0, r2.stderr.decode()[-2000:]
        assert json.loads(r2.stdout.decode().strip().split("\n")[-1])["b200"] == out["b200"], knobs
    kats = json.load(open(os.path.join(GOLDEN, "oracle_kats.json")))
    for case, o in out.items():
        g = golden_lines(case)
        a, b, c = o["text"].split("\n")[:3]
        assert b == str(g["hit_time_step"]) and c == g["text"].split("\n")[2]
        assert abs(float(a) - g["min_dist"]) <= MIN_DIST_RTOL * g["min_dist"]
        k = kats[case]
        assert o["argmin"] == k["argmin_step"]
        assert o["reach"] == [d["reach_step"] for d in k["devices"]]
        assert o["q3"] == [d["q3_hit_step"] for d in k["devices"]]


@pytest.mark.parametrize("case", ["b80", "b90", "b200"])
def test_scheduler_parts_between_two_and_trajectory_count(nb, case, kats):
    """2 < GPUs < trajectories (hw5.cu:448-457, 575-588 generalised): part 0 = query 1, part 1 = query 2 -> the query-3
    candidates it was left with, parts 2.. = speculative query-3 trajectories (from step 0) of the devices nearest to the
    planet.  The parts run one after another on this GPU and are merged exactly as solve_distributed / nb_solve do."""
    s = nb.read_input(case_path(case))
    g = golden_lines(case)
    T = 2 + len(s.devices)
    for n_parts in range(3, T):
        merged = None
        spare_entries = 0
        for part in range(n_parts):
            evs, secs, pairs = nb.solve_partial(s, 0, part, n_parts)
            if merged is None:
                merged = (nb.NbEvents * T)()
                for t in range(T):
                    merged[t].steps_done = -2
            for t in range(T):
                if evs[t].steps_done != -2:
                    assert merged[t].steps_done == -2, "a trajectory belongs to one part"
                    merged[t] = evs[t]
                    if part >= 2:
                        spare_entries += 1
                        assert t >= 2 and evs[t].steps_done >= 0
        assert spare_entries == n_parts - 2, "every spare part simulated one query-3 trajectory"
        ans = nb.solve_combine(s, merged)
        assert (ans.hit_time_step, ans.gravity_device_id, ans.missile_cost) == (
            g["hit_time_step"], g["gravity_device_id"], g["missile_cost"]), n_parts
        assert abs(ans.min_dist - g["min_dist"]) <= MIN_DIST_RTOL * g["min_dist"]
        for k, d in enumerate(kats[case]["devices"]):  # whatever was simulated agrees with the oracle's per-device outcome
            if ans.q3_hit_step[k] != -3:
                assert ans.q3_hit_step[k] == d["q3_hit_step"]


def test_grid_exchange_knobs_never_change_results_full_length(nb):
    """The fence-free exchange of the grid kernel (self-checking 32-byte records, TMA multicast, poll-and-patch) is
    timing-dependent by design; its RESULTS must not be.  b1024 and b512, all 200 000 steps, with clusters of 1 / 2 / 4,
    the copy issued with no delay at all for one system and for two in lock step (every record stale at first: all go
    through the poll-and-patch path), one or two systems per launch, a constant or a faster-moving adaptive copy delay:
    final q and v bit-identical, same events."""
    import sys
    code = ("import importlib, hashlib, json, sys\n"
            "sys.path.insert(0, %r)\n"
            "nb = importlib.import_module('nthu_ipc_nbody-simulation_b200')\n"
            "out = {}\n"
            "for case in ('b1024', 'b512'):\n"
            "    s = nb.read_input(%r + '/' + case + '.in')\n"
            "    a = nb.Trajectory(s, nb.KIND_Q1)\n"
            "    ev = a.run(nb.N_STEPS)\n"
            "    q, v, m, step = a.state()\n"
            "    out[case] = [hashlib.sha256(q.tobytes() + v.tobytes()).hexdigest(), ev.argmin_step, repr(ev.min_d2), step]\n"
            "    ans = nb.solve(s, gpus=[0])\n"
            "    out[case] += [nb.format_output(ans.min_dist, ans.hit_time_step, ans.gravity_device_id, ans.missile_cost)]\n"
            "print(json.dumps(out))\n") % (ROOT, os.path.join(GOLDEN, "testcases"))
    results = {}
    for name, knobs in (("default", {}), ("cs1", dict(NB_GRID_CS="1")), ("cs2_t1", dict(NB_GRID_CS="2", NB_GRID_T="1")),
                        ("cs4_delay0", dict(NB_GRID_CS="4", NB_GRID_DELAY="0")), ("cs2_delay0_t2", dict(NB_GRID_CS="2", NB_GRID_DELAY="0", NB_GRID_T="2")),
                        ("delay5000_constant", dict(NB_GRID_DELAY="5000", NB_GRID_ADAPT="0,0")), ("constant900", dict(NB_GRID_ADAPT="0,0")),
                        ("adapt_fast", dict(NB_GRID_ADAPT="400,100")), ("lockstep_delay0", dict(NB_GRID_DELAY2="0"))):
        r = subprocess.run([sys.executable, "-c", code], capture_output=True, env=dict(os.environ, **knobs), timeout=900)
        assert r.returncode == 0, (name, r.stderr.decode()[-2000:])
        results[name] = json.loads(r.stdout.decode().strip().split("\n")[-1])
    for name, res in results.items():
        assert res == results["default"], name
    for case in ("b1024", "b512"):
        assert results["default"][case][4] == golden_lines(case)["text"]


def test_grid_kernel_large_then_small_then_large_in_one_process(nb):
    """The dynamic shared-memory limit is an attribute of the kernel function: b1024 (160 KB), then b512 (80 KB), then
    b1024 again in ONE process must not launch against a lowered limit (round-1 advisor finding, nb_grid.cu)."""
    big, small = nb.read_input(case_path("b1024")), nb.read_input(case_path("b512"))
    ref = {}
    for name, s in (("b1024", big), ("b512", small), ("b1024", big), ("b512", small)):
        t = nb.Trajectory(s, nb.KIND_Q1)
        ev = t.run(3000)
        q = t.state()[0]
        t.close()
        if name in ref:
            assert np.array_equal(ref[name], q)
        ref[name] = q
        assert ev.steps_done == 3000


def test_grid_kernel_unavailable_falls_back_to_single_block(nb):
    """When the grid kernel's clusters cannot be co-resident (MIG / MPS / a shared GPU) the launch returns
    NB_ERR_UNSUPPORTED before anything ran and the trajectory takes the single-block kernel: same discrete answers.
    Forced here with NB_GRID_FORCE_UNSUPPORTED=1 in a subprocess."""
    import sys
    code = ("import importlib, sys\n"
            "sys.path.insert(0, %r)\n"
            "nb = importlib.import_module('nthu_ipc_nbody-simulation_b200')\n"
            "s = nb.read_input(%r)\n"
            "a = nb.solve(s, gpus=[0], n_steps=4000)\n"
            "print(a.argmin_step, '%%.16e' %% a.min_dist, a.hit_time_step)\n") % (ROOT, case_path("b200"))
    outs = []
    for env in (dict(os.environ), dict(os.environ, NB_GRID_FORCE_UNSUPPORTED="1", NB_VERBOSE="1")):
        r = subprocess.run([sys.executable, "-c", code], capture_output=True, env=env, timeout=600)
        assert r.returncode == 0, r.stderr.decode()[-2000:]
        outs.append(r.stdout.decode().strip().split("\n")[-1])
        if "NB_GRID_FORCE_UNSUPPORTED" in env:
            assert "single-block kernel instead" in r.stderr.decode()
    assert outs[0] == outs[1]


# ---- nbtool: generator / ensembles / state files from the command line (SURVEY 8f rank 4) -----------------------
def test_nbtool_ensemble_and_advance(nb, oracle, tmp_path):
    """`nbtool ensemble` = config C4's members (velocities scaled by 1 + 1e-9 k) through nb_ensemble_run over the visible
    GPUs; `nbtool advance` = run_step x steps with the state written in the reference's input format."""
    out = tmp_path / "ens.txt"
    subprocess.check_call([nb.NBTOOL_PATH, "ensemble", case_path("b100"), "5", "2000", str(out)])
    rows = [l.split() for l in out.read_text().strip().split("\n")]
    assert [int(r[0]) for r in rows] == [0, 1, 2, 3, 4]
    s = nb.read_input(case_path("b100"))
    for k in (0, 3):
        t = nb.Trajectory(nb.System(s.n, s.planet, s.asteroid, s.q, s.v * (1 + 1e-9 * k), s.m, s.is_device), nb.KIND_Q2)
        ev = t.run(2000)
        t.close()
        assert float(rows[k][1]) == float("%.16e" % np.sqrt(ev.min_d2)) and int(rows[k][2]) == ev.argmin_step and int(rows[k][3]) == ev.hit_step
    lst = tmp_path / "list.txt"
    lst.write_text("# two goldens of the same n would go here\n%s\n%s\n" % (case_path("b100"), case_path("b100")))
    out2 = tmp_path / "ens2.txt"
    subprocess.check_call([nb.NBTOOL_PATH, "ensemble-list", str(lst), "2000", str(out2)])
    rows2 = [l.split() for l in out2.read_text().strip().split("\n")]
    assert rows2[0][1:] == rows[0][1:] and rows2[1][1:] == rows[0][1:]
    adv = tmp_path / "adv.in"
    subprocess.check_call([nb.NBTOOL_PATH, "advance", case_path("b50"), "500", str(adv)])
    a = nb.read_input(str(adv))
    s = nb.read_input(case_path("b50"))
    q, v = s.q.copy(), s.v.copy()
    nb.run_steps(0, 500, s.n, q, v, s.m, s.is_device)
    assert np.array_equal(a.q, q) and np.array_equal(a.v, v)
    qo, vo = s.q.copy(), s.v.copy()
    oracle.run_steps(oracle.MODE_SQRT3, s.n, qo, vo, s.m, s.is_device, 0, 500)
    assert np.max(np.abs(a.q - qo) / np.abs(qo)) < 1e-15  # FAST kernel vs oracle after 500 steps


# ---- ensembles ---------------------------------------------------------------------------------------
def test_ensemble_members_match_individual_runs(nb, oracle):
    """SURVEY §8d config C4 in miniature: member k = the golden system with velocities scaled by (1 + 1e-9 k)."""
    s = nb.read_input(case_path("b100"))
    S, steps = 12, 300
    q = np.tile(s.q, (S, 1))
    v = np.stack([s.v * (1 + 1e-9 * k) for k in range(S)])
    m = np.tile(s.m, (S, 1))
    dev = np.tile(s.is_device, (S, 1))
    q_in, v_in = q.copy(), v.copy()
    ev, secs = nb.ensemble_run(q, v, m, dev, [s.planet] * S, [s.asteroid] * S, kind=nb.KIND_Q2, step_end=steps,
                               math=nb.MATH_STRICT)
    assert secs > 0
    for k in (0, 5, S - 1):
        qo, vo = q_in[k].copy(), v_in[k].copy()
        oracle.run_steps(oracle.MODE_SQRT3, s.n, qo, vo, s.m, s.is_device, 0, steps)
        assert np.array_equal(q[k], qo) and np.array_equal(v[k], vo)
        assert ev[k].steps_done == steps and ev[k].hit_step == -2
    assert not np.array_equal(q[1], q[2])


def test_symmetric_single_block_kernel_b1024_ensemble(nb, oracle, kats):
    """The 1024-body ensemble (config C4) runs on traj_sym_kernel (every unordered pair of different groups once).
    (1) the four trajectories of b1024 (query 1, query 2, query 3 for both devices) as ONE ensemble launch, full
    200 000 steps: events equal the oracle's known answers and the golden; (2) state after 2000 steps against the CPU
    oracle at the FAST tolerance (q within 2 ulp); (3) a 900-body system (partial last group) against the oracle."""
    s = nb.read_input(case_path("b1024"))
    devs = s.devices
    # (2) + resume in two launches
    S = 2
    q, v = np.tile(s.q, (S, 1)), np.tile(s.v, (S, 1))
    m, dev = np.tile(s.m, (S, 1)), np.tile(s.is_device, (S, 1))
    ev, _ = nb.ensemble_run(q, v, m, dev, [s.planet] * S, [s.asteroid] * S, kind=nb.KIND_Q2, step_end=2000)
    qo, vo = s.q.copy(), s.v.copy()
    oracle.run_steps(oracle.MODE_SQRT3, s.n, qo, vo, s.m, s.is_device, 0, 2000)
    assert ulps(q[0], qo).max() <= 2 and np.allclose(v[0], vo, rtol=1e-12, atol=0)
    assert np.array_equal(q[0], q[1]) and ev[0].steps_done == 2000
    # (3) ragged
    r = nb.synthetic_system(900, seed=5)
    q, v = r.q.copy()[None], r.v.copy()[None]
    nb.ensemble_run(q, v, r.m[None], r.is_device[None], [0], [1], kind=nb.KIND_PLAIN, step_end=50)
    qo, vo = r.q.copy(), r.v.copy()
    oracle.run_steps(oracle.MODE_SQRT3, r.n, qo, vo, r.m, r.is_device, 0, 50)
    assert ulps(q[0], qo).max() <= 2 and np.allclose(v[0], vo, rtol=1e-12, atol=0)
    # (1) full length, one launch for each kind (kinds are per launch)
    k = kats["b1024"]
    g = golden_lines("b1024")
    one = lambda a: a.copy()[None]
    e1, _ = nb.ensemble_run(one(s.q), one(s.v), one(np.where(s.is_device, 0.0, s.m)), one(s.is_device), [s.planet], [s.asteroid],
                            kind=nb.KIND_Q1, step_end=nb.N_STEPS)
    assert e1[0].argmin_step == k["argmin_step"] and abs(np.sqrt(e1[0].min_d2) - g["min_dist"]) <= MIN_DIST_RTOL * g["min_dist"]
    e2, _ = nb.ensemble_run(one(s.q), one(s.v), one(s.m), one(s.is_device), [s.planet], [s.asteroid], kind=nb.KIND_Q2,
                            step_end=nb.N_STEPS)
    assert e2[0].hit_step == g["hit_time_step"]
    assert list(e2[0].reach_step[:len(devs)]) == [d["reach_step"] for d in k["devices"]]
    S = len(devs)
    e3, _ = nb.ensemble_run(np.tile(s.q, (S, 1)), np.tile(s.v, (S, 1)), np.tile(s.m, (S, 1)), np.tile(s.is_device, (S, 1)),
                            [s.planet] * S, [s.asteroid] * S, kind=nb.KIND_Q3, destroy_device=devs, step_end=nb.N_STEPS)
    for i, d in enumerate(k["devices"]):
        assert e3[i].hit_step == d["q3_hit_step"] and e3[i].destroyed_step == d["reach_step"]
    saved = [(e3[i].cost, devs[i]) for i in range(S) if e3[i].hit_step == -2]
    assert min(saved)[1] == g["gravity_device_id"] and min(saved)[0] == g["missile_cost"]


# ---- large-N path ------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [1025, 3000, 4096])
def test_large_path_strict_bitwise(nb, oracle, n):
    """n > 1024 goes through the tiled TMA kernel; STRICT sums j ascending in one split -> bit-identical."""
    s = nb.synthetic_system(n, seed=3)
    q, v = s.q.copy(), s.v.copy()
    nb.run_steps(0, 3, n, q, v, s.m, s.is_device, math=nb.MATH_STRICT)
    qo, vo = s.q.copy(), s.v.copy()
    oracle.run_steps(oracle.MODE_SQRT3, n, qo, vo, s.m, s.is_device, 0, 3)
    assert np.array_equal(q, qo) and np.array_equal(v, vo)


def test_large_path_fast_accelerations(nb, oracle):
    """SURVEY §8d C5 parity: after one step from rest v = a*dt; every component within 1e-12 of the
    body's largest acceleration component; after 10 steps q within 1e-12*max|v|*dt, v within 1e-12."""
    n = 8192
    s = nb.synthetic_system(n, seed=42)
    rest = s.copy()
    rest.v[:] = 0.0
    q, v = rest.q.copy(), rest.v.copy()
    nb.run_steps(0, 1, n, q, v, rest.m, rest.is_device)
    qo, vo = rest.q.copy(), rest.v.copy()
    oracle.run_steps(oracle.MODE_STRICT, n, qo, vo, rest.m, rest.is_device, 0, 1)
    scale = np.abs(vo.reshape(3, -1)).max(axis=0)
    assert (np.abs(v - vo).reshape(3, -1) / scale).max() < 1e-12
    q, v = s.q.copy(), s.v.copy()
    nb.run_steps(0, 10, n, q, v, s.m, s.is_device)
    qo, vo = s.q.copy(), s.v.copy()
    oracle.run_steps(oracle.MODE_SQRT3, n, qo, vo, s.m, s.is_device, 0, 10)
    assert np.abs(q - qo).max() <= max(1e-12 * np.abs(vo).max() * 60.0, 2 * np.spacing(np.abs(qo)).max())
    assert np.allclose(v, vo, rtol=1e-12, atol=0)


def test_full_size_65536_one_step_against_oracle_and_invariants(nb, oracle):
    """BASELINE's full size (config C5, 65 536 bodies): one step from rest, so v = a*dt.
    (1) against the CPU oracle (all host threads, 4.3e9 pairs): every component within 1e-12 of the body's
        largest component; (2) momentum: sum_i m_i a_i = 0 for exact pairwise forces (Newton's third law) - a
        checksum over all 4.3e9 pair terms that needs no oracle; (3) linearity: doubling every mass doubles
        every acceleration bit for bit (power-of-two scaling commutes with every rounding)."""
    n = 65536
    s = nb.synthetic_system(n, seed=42)
    s.v[:] = 0.0
    s.is_device[:] = 0  # the modulation is covered elsewhere; here G*m is a pure per-body scale
    q, v = s.q.copy(), s.v.copy()
    nb.run_steps(0, 1, n, q, v, s.m, s.is_device)
    qo, vo = s.q.copy(), s.v.copy()
    oracle.run_steps(oracle.MODE_SQRT3, n, qo, vo, s.m, s.is_device, 0, 1)
    scale = np.abs(vo.reshape(3, -1)).max(axis=0)
    assert (np.abs(v - vo).reshape(3, -1) / scale).max() < 1e-12
    assert np.abs(q - qo).max() <= 2 * np.spacing(np.abs(qo)).max()
    a = v.reshape(3, n) / 60.0
    p = (a * s.m).sum(axis=1)
    assert np.all(np.abs(p) <= 1e-11 * np.abs(a * s.m).sum(axis=1))
    q2, v2 = s.q.copy(), s.v.copy()
    nb.run_steps(0, 1, n, q2, v2, 2.0 * s.m, s.is_device)
    assert np.array_equal(v2, 2.0 * v)


def close_states(q, v, qo, vo):
    """FAST-math tolerance of SURVEY 8d C5: q within 1e-12*max|v|*dt (or 2 ulp), v within 1e-12 relative."""
    return (np.abs(q - qo).max() <= max(1e-12 * np.abs(vo).max() * 60.0, 2 * np.spacing(np.abs(qo)).max())
            and np.allclose(v, vo, rtol=1e-12, atol=0))


def test_sharded_single_rank_matches_host_api(nb):
    """The torch-plumbed device-pointer paths against nb_run_steps (which takes the symmetric stepper for FAST math):
    SymShardedSystem is the same kernels -> bit for bit; ShardedSystem (row kernel, nb_large_pack / nb_large_step)
    sums in another order -> FAST tolerance."""
    import torch

    n = 4096
    s = nb.synthetic_system(n, seed=11)
    q, v = s.q.copy(), s.v.copy()
    nb.run_steps(0, 5, n, q, v, s.m, s.is_device)
    sy = nb.SymShardedSystem(s, rank=0, world=1, device="cuda:0")
    sy.advance(5)
    assert np.array_equal(sy.positions(), q) and np.array_equal(sy.velocities(), v)
    sy.close()
    sh = nb.ShardedSystem(s, rank=0, world=1, device="cuda:0")
    sh.advance(5)
    torch.cuda.synchronize()
    assert close_states(sh.positions(), sh.velocities(), q, v)


@pytest.mark.parametrize("n,world", [(6144, 2), (6144, 3), (6144, 4), (8192, 8), (3000, 1), (5000, 2)])
def test_symmetric_stepper_multi_rank_on_one_gpu(nb, oracle, n, world):
    """The multi-rank path of the symmetric stepper (block-pair assignment, partial rows stored into the owner's PJ,
    arrival counters, in-kernel waits, pos4 rows stored into every rank) with all ranks on this GPU (SymLocalWorld):
    against the CPU oracle at the FAST tolerance, run to run bit-identical, and no wait timed out (positions() checks
    the status word).  Ragged shards (1500 = 1024 + 476 bodies) included."""
    s = nb.synthetic_system(n, seed=17)
    steps = 6
    w = nb.SymLocalWorld(s, world, device="cuda:0")
    w.advance(steps)
    q, v = w.positions(), w.velocities()
    for r in w.ranks[1:]:
        assert np.array_equal(r.positions(), q), "every rank holds the same positions"
    w.close()
    qo, vo = s.q.copy(), s.v.copy()
    oracle.run_steps(oracle.MODE_SQRT3, n, qo, vo, s.m, s.is_device, 0, steps)
    assert close_states(q, v, qo, vo)
    w2 = nb.SymLocalWorld(s, world, device="cuda:0")
    w2.advance(steps)
    assert np.array_equal(w2.positions(), q) and np.array_equal(w2.velocities(), v), "deterministic"
    w2.close()


def test_symmetric_stepper_accelerations_ragged(nb, oracle):
    """One step from rest (v = a*dt) on sizes that leave partial rows, partial j tiles and partial rotation groups."""
    for n in (1025, 1500, 2049, 3333):
        s = nb.synthetic_system(n, seed=n)
        s.v[:] = 0.0
        q, v = s.q.copy(), s.v.copy()
        nb.run_steps(0, 1, n, q, v, s.m, s.is_device)
        qo, vo = s.q.copy(), s.v.copy()
        oracle.run_steps(oracle.MODE_STRICT, n, qo, vo, s.m, s.is_device, 0, 1)
        scale = np.abs(vo.reshape(3, -1)).max(axis=0)
        assert (np.abs(v - vo).reshape(3, -1) / scale).max() < 1e-12, n


def test_p2p_fused_exchange_single_rank(nb):
    """The integrate kernel that stores the new rows into the peers' buffers (here: only its own) and the
    counter / device-side wait protocol give the NCCL path's result bit for bit."""
    import torch

    n = 4096
    s = nb.synthetic_system(n, seed=11)
    a = nb.ShardedSystem(s, device="cuda:0")
    b = nb.P2PShardedSystem(s, device="cuda:0")
    a.advance(7)
    b.advance(7)
    torch.cuda.synchronize()
    assert np.array_equal(a.positions(), b.positions()) and np.array_equal(a.velocities(), b.velocities())
    b.close()


def test_two_shards_on_one_gpu_equal_one_shard(nb):
    """Body sharding is exact: integrating [0, n/2) and [n/2, n) separately against all bodies and
    exchanging pos4 rows gives the unsharded result bit for bit (the all-gather is emulated by a copy)."""
    import torch

    n = 2048
    s = nb.synthetic_system(n, seed=5)
    whole = nb.ShardedSystem(s, rank=0, world=1, device="cuda:0")
    parts = [nb.ShardedSystem(s, rank=r, world=2, device="cuda:0") for r in range(2)]
    for p in parts:
        p.world = 1  # no process group here: the exchange is done by hand below
    for _ in range(4):
        whole.advance(1)
        for p in parts:
            p.advance(1)
        a, b = parts
        h = n // 2
        a.pos4[a.cur][h:] = b.pos4[b.cur][h:]
        b.pos4[b.cur][:h] = a.pos4[a.cur][:h]
    torch.cuda.synchronize()
    assert torch.equal(whole.pos4[whole.cur], parts[0].pos4[parts[0].cur])
    assert torch.equal(whole.pos4[whole.cur], parts[1].pos4[parts[1].cur])
    assert torch.equal(whole.vel[:, : n // 2], parts[0].vel) and torch.equal(whole.vel[:, n // 2:], parts[1].vel)


def test_fp64_peak_is_plausible(nb):
    tf = nb.fp64_peak(0)
    assert 15.0 < tf < 45.0, tf
