"""GPU: nb_ensemble_run for systems of more than 1024 bodies (nb_ens.cu: one pair-kernel launch per step for a whole group of
systems, DeviceBatch::run_ens_large in nb_host.cu).

Tile edge 128: the tiling edges are the first and last body of each 128-body tile, the ragged last tile and the diagonal
tiles.  STRICT sums j in ascending order, so it is the oracle's SQRT3 mode to the bit; FAST is held to the FAST tolerance
of the oracle and to the sparse-source bound of the exact accelerations."""
import math
import subprocess

import numpy as np
import pytest
from conftest import case_path
from test_gpu_large_queries import check_golden, collision_system, discrete, fields, kats, padded  # noqa: F401
from test_gpu_pair_error_bound import check_bound, gm_of, sparse_system

pytestmark = pytest.mark.gpu
STEPS = 1000  # horizon of the constructed collision systems


def close_states(q, v, qo, vo):
    """FAST-math tolerance of SURVEY 8d C5: q within 1e-12*max|v|*dt (or 2 ulp), v within 1e-12 relative."""
    return (np.abs(q - qo).max() <= max(1e-12 * np.abs(vo).max() * 60.0, 2 * np.spacing(np.abs(qo)).max())
            and np.allclose(v, vo, rtol=1e-12, atol=0))


def stack(systems):
    return (np.stack([s.q for s in systems]), np.stack([s.v for s in systems]), np.stack([s.m for s in systems]),
            np.stack([s.is_device for s in systems]))


def run(nb, systems, step_end, kind=0, math_=0, destroy=None, step_begin=0):
    """ensemble_run on copies of the systems' arrays -> (q [S, 3n], v [S, 3n], events)."""
    q, v, m, dev = stack(systems)
    ev, _ = nb.ensemble_run(q, v, m, dev, [s.planet for s in systems], [s.asteroid for s in systems], kind=kind,
                            destroy_device=destroy, step_begin=step_begin, step_end=step_end, math=math_)
    return q, v, ev


def synthetic(nb, n, seeds):
    return [nb.generate_system(n, seed=int(k)) for k in seeds]


def colliding(nb, n):
    """Three collision systems whose planet and asteroid start 1, 0.8 and 0.7 times as far apart: at n = 1025 the oracle
    (SQRT3) has them hit at steps 476, 401 and 347."""
    out = []
    for f in (1.0, 0.8, 0.7):
        s = collision_system(nb, n)
        s.q[s.planet] *= f
        s.q[s.asteroid] *= f
        out.append(s)
    return out


# ---- state against the oracle ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [1025, 2049, 3333])
def test_strict_is_bitwise_the_oracle(nb, oracle, n):
    systems = synthetic(nb, n, [n, n + 1, n + 2])
    q, v, ev = run(nb, systems, 5, math_=nb.MATH_STRICT)
    for k, s in enumerate(systems):
        qo, vo = s.q.copy(), s.v.copy()
        oracle.run_steps(oracle.MODE_SQRT3, n, qo, vo, s.m, s.is_device, 0, 5)
        assert ev[k].steps_done == 5
        assert np.array_equal(q[k], qo) and np.array_equal(v[k], vo), (n, k)


@pytest.mark.parametrize("n", [1025, 2049, 3333, 8192])
def test_fast_within_tolerance_of_the_oracle(nb, oracle, n):
    systems = synthetic(nb, n, [7 * n, 7 * n + 1, 7 * n + 2])
    q, v, ev = run(nb, systems, 10)
    for k, s in enumerate(systems):
        qo, vo = s.q.copy(), s.v.copy()
        oracle.run_steps(oracle.MODE_SQRT3, n, qo, vo, s.m, s.is_device, 0, 10)
        assert ev[k].steps_done == 10
        assert close_states(q[k], v[k], qo, vo), (n, k)


# sources on the tile edges: first and last body of tiles, the ragged last tile, both ends of diagonal tiles
EDGES = [
    (1025, [0, 127, 128, 255, 256, 511, 512, 895, 896, 1023, 1024]),
    (2049, [0, 1, 127, 128, 1023, 1024, 1151, 1152, 1919, 1920, 2047, 2048]),
    (3333, [0, 127, 128, 1791, 1792, 3071, 3072, 3073, 3199, 3200, 3327, 3328, 3332]),
]


@pytest.mark.parametrize("n,sources", EDGES, ids=[str(c[0]) for c in EDGES])
def test_sparse_sources_on_tile_edges(nb, n, sources):
    """One step from rest, two systems in one launch (the second with its sources mirrored), each with one heavy gravity
    device: every component within (K + k) u dt sum|term| of the exact acceleration."""
    systems = [sparse_system(nb, n, sources, seed=n), sparse_system(nb, n, [n - 1 - j for j in sources], seed=n + 1)]
    assert all(s.is_device.sum() == 1 for s in systems)
    _, v, ev = run(nb, systems, 1)
    assert all(e.steps_done == 1 for e in ev)
    for k, s in enumerate(systems):
        check_bound(v[k], s.q, gm_of(s.m, s.is_device, 1), "ensemble n=%d system %d" % (n, k))


# ---- a member's result depends on its own inputs only ---------------------------------------------------------------
def test_members_independent_of_the_batch_and_deterministic(nb):
    """A mixed Q2 batch: three collision systems that hit (and stop) at different steps, four synthetic systems that do
    not.  Each member equals the same system run alone, and a second call, bit for bit."""
    n = 1025
    systems = colliding(nb, n) + synthetic(nb, n, [11, 12, 13, 14])
    order = [3, 0, 4, 1, 5, 2, 6]
    systems = [systems[i] for i in order]
    q, v, ev = run(nb, systems, 600, kind=nb.KIND_Q2)
    hits = [e.hit_step for e in ev]
    assert len({h for h in hits if h != -2}) >= 2 and [hits[i] for i in (0, 2, 4, 6)] == [-2] * 4, hits
    q2, v2, ev2 = run(nb, systems, 600, kind=nb.KIND_Q2)
    assert np.array_equal(q, q2) and np.array_equal(v, v2)
    assert [e.as_dict() for e in ev] == [e.as_dict() for e in ev2]
    for k, s in enumerate(systems):
        qs, vs, es = run(nb, [s], 600, kind=nb.KIND_Q2)
        assert np.array_equal(q[k], qs[0]) and np.array_equal(v[k], vs[0]), k
        assert ev[k].as_dict() == es[0].as_dict(), k


def test_groups_give_the_solo_results(nb):
    """Six systems of 65 536 bodies do not fit one group's scratch budget (2 GiB: two systems of 809 MB), so they run as
    three groups, which the launch count shows: per group one observer launch for step 0 and three launches per step,
    plus one pack and one unpack per system.  Every member equals its solo run bit for bit."""
    n, S, steps = 65536, 6, 2
    systems = synthetic(nb, n, range(100, 100 + S))
    before = nb.kernel_launches()
    q, v, ev = run(nb, systems, steps)
    assert nb.kernel_launches() - before == S + 3 * (1 + 3 * steps) + S
    for k, s in enumerate(systems):
        qs, vs, _ = run(nb, [s], steps)
        assert np.array_equal(q[k], qs[0]) and np.array_equal(v[k], vs[0]), k


# ---- events ---------------------------------------------------------------------------------------------------------
def ensemble_answer(nb, s, n_steps, math_):
    """The three queries as three ensemble launches (Q1, Q2, and Q3 with every device destroyed in turn), combined by
    the library's selection rule.  Returns (answer, Q2 events, Q3 events)."""
    _, _, e1 = run(nb, [s], n_steps, kind=nb.KIND_Q1, math_=math_)
    _, _, e2 = run(nb, [s], n_steps, kind=nb.KIND_Q2, math_=math_)
    devs = s.devices
    _, _, e3 = run(nb, [s] * len(devs), n_steps, kind=nb.KIND_Q3, math_=math_, destroy=devs)
    evs = (nb.NbEvents * (2 + len(devs)))(*([e1[0], e2[0]] + list(e3)))
    return nb.solve_combine(s, evs), e2[0], e3


@pytest.mark.parametrize("n", [1025, 2049])
def test_events_against_the_oracle(nb, oracle, n):
    s = collision_system(nb, n)
    ref = oracle.solve(oracle.MODE_SQRT3, s, n_steps=STEPS)
    assert ref.hit_time_step == 476 and ref.gravity_device_id == 3
    ans, q2, q3 = ensemble_answer(nb, s, STEPS, nb.MATH_STRICT)
    assert fields(ans) == fields(ref)
    for k, e in enumerate(q3):
        assert e.destroyed_step == q2.reach_step[k] != -2, k
    ans, _, _ = ensemble_answer(nb, s, STEPS, nb.MATH_FAST)
    assert discrete(ans) == discrete(ref)


def test_stopped_members_return_their_hit_state(nb, oracle):
    """STRICT Q2: members that hit at different steps come back with q, v of their own hit step."""
    n = 1025
    systems = colliding(nb, n)
    q, v, ev = run(nb, systems, STEPS, kind=nb.KIND_Q2, math_=nb.MATH_STRICT)
    hits = [e.hit_step for e in ev]
    assert hits == [476, 401, 347], hits
    for k, s in enumerate(systems):
        assert ev[k].steps_done == hits[k]
        qo, vo = s.q.copy(), s.v.copy()
        oracle.run_steps(oracle.MODE_SQRT3, n, qo, vo, s.m, s.is_device, 0, hits[k])
        assert np.array_equal(q[k], qo) and np.array_equal(v[k], vo), k


def test_resume(nb):
    """FAST Q2, 0 -> 300 then 300 -> 700 against 0 -> 700: the same state at the hit step (476) and the same events
    (minimum distance and reach steps taken over both calls)."""
    s = collision_system(nb, 1025)
    qf, vf, ef = run(nb, [s], 700, kind=nb.KIND_Q2)
    qa, va, ea = run(nb, [s], 300, kind=nb.KIND_Q2)
    part = s.copy()
    part.q, part.v = qa[0].copy(), va[0].copy()
    qb, vb, eb = run(nb, [part], 700, kind=nb.KIND_Q2, step_begin=300)
    assert ea[0].steps_done == 300 and ea[0].hit_step == -2
    assert ef[0].hit_step == eb[0].hit_step == eb[0].steps_done == ef[0].steps_done == 476
    assert np.array_equal(qf, qb) and np.array_equal(vf, vb)
    a, b, f = ea[0], eb[0], ef[0]
    first = (a.min_d2, a.argmin_step) if a.min_d2 <= b.min_d2 else (b.min_d2, b.argmin_step)
    assert first == (f.min_d2, f.argmin_step)
    reach = [x if x != -2 else y for x, y in zip(a.reach_step[:a.n_reach], b.reach_step[:b.n_reach])]
    assert reach == list(f.reach_step[:f.n_reach])


@pytest.mark.parametrize("case,n", [("b100", 1025), ("b1024", 2048)])
def test_padded_goldens_full_length(nb, kats, case, n):
    s = padded(nb, case, n)
    ans, _, _ = ensemble_answer(nb, s, 200000, nb.MATH_FAST)
    check_golden(ans, case, kats)


# ---- CLI, arguments, routing --------------------------------------------------------------------------------------
def test_nbtool_ensemble_above_1024(nb, tmp_path):
    inp, out = tmp_path / "b100_1025.in", tmp_path / "members.txt"
    nb.write_input(str(inp), padded(nb, "b100", 1025))
    subprocess.check_call([nb.NBTOOL_PATH, "ensemble", str(inp), "3", "400", str(out)])
    lines = out.read_text().splitlines()
    assert len(lines) == 3
    s = nb.read_input(str(inp))
    _, _, ev = run(nb, [s], 400, kind=nb.KIND_Q2)
    e = ev[0]
    assert lines[0] == "0 %.16e %d %d" % (math.sqrt(e.min_d2), e.argmin_step, e.hit_step)


def test_argument_and_limit_checks(nb):
    s = collision_system(nb, 1025)
    with pytest.raises(nb.NbodyError) as e:
        run(nb, [s], 10, kind=nb.KIND_Q3)
    assert e.value.code == nb.NB_ERR_ARG
    with pytest.raises(nb.NbodyError) as e:
        run(nb, [collision_system(nb, 1025, n_dev=65)], 10)
    assert e.value.code == nb.NB_ERR_UNSUPPORTED
    with pytest.raises(nb.NbodyError) as e:
        run(nb, [collision_system(nb, 65537)], 1)
    assert e.value.code == nb.NB_ERR_UNSUPPORTED


# Run in a process of its own: a CUDA profiler session leaves the profiling library attached to the process, and the
# kernel records of later sessions in the same process (test_gpu_pair_error_bound's routing test) can then go missing.
ROUTING = r"""
import importlib, json, sys
sys.path.insert(0, sys.argv[1])
import numpy as np
from torch.profiler import ProfilerActivity, profile
nb = importlib.import_module("nthu_ipc_nbody-simulation_b200")
out = {}
for label, n, S, steps, math_ in (("fast", 2048, 4, 5, nb.MATH_FAST), ("strict", 2048, 4, 5, nb.MATH_STRICT),
                                  ("small", 1024, 2, 2, nb.MATH_FAST)):
    systems = [nb.generate_system(n, seed=k) for k in range(S)]
    q, v = np.stack([s.q for s in systems]), np.stack([s.v for s in systems])
    m, dev = np.stack([s.m for s in systems]), np.stack([s.is_device for s in systems])
    before = nb.kernel_launches()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        nb.ensemble_run(q, v, m, dev, [s.planet for s in systems], [s.asteroid for s in systems], step_end=steps,
                        math=math_)
    out[label] = dict(launches=nb.kernel_launches() - before, kernels=[e.name for e in prof.events()])
print(json.dumps(out))
"""


def test_routing(nb):
    """n > 1024: three launches per step for the whole batch on the new kernels (plus one pack and one unpack per system
    and the observers of step 0); n = 1024 still runs traj_sym_kernel, one launch."""
    import json
    import os
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-s", "-c", ROUTING, root], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    out = json.loads(r.stdout.strip().splitlines()[-1])
    S, steps = 4, 5
    for label, pair_kernel in (("fast", "sym_ens_tile_kernel"), ("strict", "large_ens_strict_kernel")):
        assert out[label]["launches"] == S + 1 + 3 * steps + S, out[label]["launches"]
        names = [x for x in out[label]["kernels"] if "_ens_" in x]
        for k in (pair_kernel, "large_ens_integrate_kernel"):
            assert sum(k in x for x in names) == steps, (label, k, names)
        assert sum("large_ens_observe_kernel" in x for x in names) == steps + 1, (label, names)
    small = out["small"]
    assert small["launches"] == 1
    assert any("traj_sym_kernel" in x for x in small["kernels"]), small["kernels"]
    assert not any("_ens_" in x for x in small["kernels"]), small["kernels"]
