"""GPU: the three queries for systems of more than 1024 bodies (DeviceBatch::run_large in nb_host.cu: the large-N steppers
with large_observe_kernel after every step).

Two kinds of input:
  * the goldens padded past 1024 bodies with massless probes at rest, far outside the system: a probe adds only exact
    zeros to the golden bodies' forces, so the answers are the goldens' (min_dist to the FAST tolerance);
  * constructed systems whose events fall within 1 000 steps, so that the CPU oracle can check every field: a planet and
    an asteroid head on, light gravity devices nearby and one heavy device above the midpoint that pulls the two together
    (Q2 hits at step 476); with the heavy device destroyed, the hit comes after the horizon."""
import json
import os
import subprocess

import numpy as np
import pytest
from conftest import GOLDEN, case_path, golden_lines

pytestmark = pytest.mark.gpu
MIN_DIST_RTOL = 1e-6
PADDED = [("b20", 1025), ("b100", 1025), ("b512", 1500), ("b1024", 2048)]
STEPS = 1000  # horizon of the constructed systems
MAX_CHUNK = 512  # largest chunk of steps DeviceBatch::run_large enqueues between two reads of the events (run_chunks)


@pytest.fixture(scope="module")
def kats():
    return json.load(open(os.path.join(GOLDEN, "oracle_kats.json")))


def padded(nb, case, n):
    """Golden `case` with massless, non-device probes appended up to n bodies; every body keeps its index.  The probes are
    at rest on a line at 2 to 3 thousand extents of the golden system from its bounding box."""
    s = nb.read_input(case_path(case))
    k = n - s.n
    q = s.q.reshape(3, -1)
    lo, hi = q.min(axis=1), q.max(axis=1)
    extent = (hi - lo).max()
    probes = np.empty((3, k))
    probes[0] = hi[0] + extent * (2e3 + 1e3 * np.arange(k) / k)
    probes[1] = 0.5 * (lo[1] + hi[1])
    probes[2] = 0.5 * (lo[2] + hi[2])
    cat = lambda a, b: np.ascontiguousarray(np.concatenate([a, b], axis=1).reshape(-1))
    return nb.System(n, s.planet, s.asteroid, cat(q, probes), cat(s.v.reshape(3, -1), np.zeros((3, k))),
                     np.concatenate([s.m, np.zeros(k)]), np.concatenate([s.is_device, np.zeros(k, dtype=np.uint8)]))


def collision_system(nb, n, n_dev=2, seed=0):
    """Body 0 = planet, 1 = asteroid (equal masses, head on along x); bodies 2 .. n_dev light devices whose missiles
    arrive within ~120 steps; body n_dev + 1 the heavy device above the midpoint, the last of the device list; the rest
    light bodies far away, which take part in every force sum."""
    rng = np.random.default_rng(seed)
    q, v, m = np.zeros((3, n)), np.zeros((3, n)), np.zeros(n)
    dev = np.zeros(n, dtype=np.uint8)
    L, u = 5e9, 2e4
    q[0, 0], v[0, 0], m[0] = L, -u, 1e27
    q[0, 1], v[0, 1], m[1] = -L, u, 1e27
    heavy = n_dev + 1
    for i in range(2, heavy):
        q[:, i] = [L + rng.uniform(-4e9, 4e9), rng.uniform(-4e9, 4e9), rng.uniform(-4e9, 4e9)]
        m[i], dev[i] = 1e20, 1
    q[:, heavy] = [0.0, 0.0, 3e9]
    m[heavy], dev[heavy] = 3e30, 1
    k = n - heavy - 1
    q[:, heavy + 1:] = np.array([3e13, 0.0, 0.0])[:, None] + rng.uniform(-5e11, 5e11, (3, k))
    v[:, heavy + 1:] = rng.normal(0.0, 1e3, (3, k))
    m[heavy + 1:] = 10 ** rng.uniform(18, 20, k)
    return nb.System(n, 0, 1, np.ascontiguousarray(q.reshape(-1)), np.ascontiguousarray(v.reshape(-1)), m, dev)


def check_golden(ans, case, kats):
    g = golden_lines(case)
    assert (ans.hit_time_step, ans.gravity_device_id, ans.missile_cost) == (g["hit_time_step"], g["gravity_device_id"],
                                                                            g["missile_cost"])
    assert abs(ans.min_dist - g["min_dist"]) <= MIN_DIST_RTOL * g["min_dist"]
    k = kats[case]
    assert ans.argmin_step == k["argmin_step"]
    for j, d in enumerate(k["devices"]):
        assert ans.device_index[j] == d["index"]
        assert ans.reach_step[j] == d["reach_step"]
        if ans.q3_hit_step[j] != -3:  # simulated (the chain plan stops at the first saviour)
            assert ans.q3_hit_step[j] == d["q3_hit_step"]


def fields(a):
    nd = a.n_devices
    return dict(min_dist=a.min_dist, argmin_step=a.argmin_step, hit_time_step=a.hit_time_step,
                gravity_device_id=a.gravity_device_id, missile_cost=a.missile_cost, n_devices=nd,
                device_index=list(a.device_index[:nd]), reach_step=list(a.reach_step[:nd]),
                q3_hit_step=list(a.q3_hit_step[:nd]), q3_cost=list(a.q3_cost[:nd]))


def discrete(a):
    f = fields(a)
    del f["min_dist"]
    return f


# ---- padded goldens, FAST, 200 000 steps ---------------------------------------------------------------
@pytest.mark.parametrize("all_devices", [False, True], ids=["chain", "independent"])
@pytest.mark.parametrize("case,n", PADDED)
def test_padded_golden(nb, kats, case, n, all_devices):
    s = padded(nb, case, n)
    assert s.devices == nb.read_input(case_path(case)).devices
    check_golden(nb.solve(s, gpus=[0], all_devices=all_devices), case, kats)


def test_hw5_binary_on_padded_b1024(nb, tmp_path):
    inp, out = tmp_path / "b1024_2048.in", tmp_path / "b1024_2048.out"
    nb.write_input(str(inp), padded(nb, "b1024", 2048))
    r = subprocess.run([nb.HW5_PATH, str(inp), str(out)], capture_output=True)
    assert r.returncode == 0, r.stderr
    g = golden_lines("b1024")
    a, b, c = out.read_text().split("\n")[:3]
    assert b == str(g["hit_time_step"]) and c == g["text"].split("\n")[2]
    assert abs(float(a) - g["min_dist"]) <= MIN_DIST_RTOL * g["min_dist"]


# ---- constructed systems against the oracle --------------------------------------------------------------
@pytest.fixture(scope="module")
def constructed(nb, oracle):
    cache = {}

    def get(n):
        if n not in cache:
            s = collision_system(nb, n)
            cache[n] = s, oracle.solve(oracle.MODE_SQRT3, s, n_steps=STEPS)
        return cache[n]
    return get


@pytest.mark.parametrize("n", [1025, 2049, 3333])
def test_strict_equals_oracle(nb, constructed, n):
    s, ref = constructed(n)
    assert ref.hit_time_step == 476 and ref.gravity_device_id == 3  # the case is what it was built to be
    want = fields(ref)
    assert fields(nb.solve(s, gpus=[0], n_steps=STEPS, math=nb.MATH_STRICT, all_devices=True)) == want
    chain = fields(nb.solve(s, gpus=[0], n_steps=STEPS, math=nb.MATH_STRICT))
    for j, h in enumerate(chain["q3_hit_step"]):  # the chain plan simulates the candidates up to the first saviour
        if h == -3:
            want["q3_hit_step"][j], want["q3_cost"][j] = -3, float("inf")
    assert chain == want


@pytest.mark.parametrize("n", [1025, 2049, 3333])
def test_fast_matches_oracle(nb, constructed, n):
    s, ref = constructed(n)
    ans = nb.solve(s, gpus=[0], n_steps=STEPS, all_devices=True)
    assert discrete(ans) == discrete(ref)
    assert abs(ans.min_dist - ref.min_dist) <= MIN_DIST_RTOL * ref.min_dist


def test_64_devices(nb, oracle):
    """Two devices per lane of the observer warp: every Q2 reach step, and the Q3 of device 63 (the heavy one, second half
    of the list), against the oracle's trajectories."""
    s = collision_system(nb, 2048, n_dev=64)
    assert len(s.devices) == 64
    ans = nb.solve(s, gpus=[0], n_steps=STEPS, math=nb.MATH_STRICT, all_devices=True)
    q2, _, _ = oracle.trajectory(oracle.MODE_SQRT3, oracle.KIND_Q2, s, n_steps=STEPS)
    assert ans.hit_time_step == q2.hit_step == 476
    assert list(ans.reach_step[:64]) == list(q2.reach_step[:64])
    q3, _, _ = oracle.trajectory(oracle.MODE_SQRT3, oracle.KIND_Q3, s, s.devices[63], n_steps=STEPS)
    assert q3.hit_step == -2 and q3.destroyed_step != -2
    assert (ans.q3_hit_step[63], ans.q3_cost[63]) == (q3.hit_step, q3.cost)
    assert (ans.gravity_device_id, ans.missile_cost) == (s.devices[63], q3.cost)


def test_edge_cases(nb, oracle):
    base = collision_system(nb, 1025)
    nodev = base.copy()
    nodev.is_device[:] = 0
    crash = base.copy()
    for k in range(3):
        crash.q[k * crash.n + crash.asteroid] = crash.q[k * crash.n + crash.planet] + 1.0e6
    for name, s, n_steps in (("zero steps", base, 0), ("one step", base, 1), ("hit at step 0", crash, 50),
                             ("no devices", nodev, 600)):
        ref = oracle.solve(oracle.MODE_SQRT3, s, n_steps=n_steps)
        for all_devices in (False, True):
            ans = nb.solve(s, gpus=[0], n_steps=n_steps, all_devices=all_devices)
            assert (ans.hit_time_step, ans.gravity_device_id, ans.missile_cost, ans.argmin_step) == (
                ref.hit_time_step, ref.gravity_device_id, ref.missile_cost, ref.argmin_step), (name, all_devices)
            assert abs(ans.min_dist - ref.min_dist) <= MIN_DIST_RTOL * ref.min_dist, (name, all_devices)
    many = collision_system(nb, 1025, n_dev=65)
    for all_devices in (False, True):
        with pytest.raises(nb.NbodyError) as e:
            nb.solve(many, gpus=[0], n_steps=10, all_devices=all_devices)
        assert e.value.code == nb.NB_ERR_UNSUPPORTED


def test_scheduler_parts(nb):
    """Every split of the trajectories into 2 .. T parts, run one after another on GPU 0 and merged as solve_distributed
    does, gives nb.solve's answer."""
    s = collision_system(nb, 1025)
    T = 2 + len(s.devices)
    want = fields(nb.solve(s, gpus=[0], n_steps=STEPS))
    for n_parts in range(2, T + 1):
        merged = (nb.NbEvents * T)()
        for t in range(T):
            merged[t].steps_done = -2
        for part in range(n_parts):
            evs, _, _ = nb.solve_partial(s, 0, part, n_parts, n_steps=STEPS)
            for t in range(T):
                if evs[t].steps_done != -2:
                    merged[t] = evs[t]
        assert fields(nb.solve_combine(s, merged)) == want, n_parts


def test_stepping_stops_after_the_hit(nb):
    """Q2 alone (independent plan, one trajectory per part) hits at step 476 of 20 000: stepping ends within the two
    chunks in flight after the hit.  A FAST step is three launches (acceleration, integrate, observer)."""
    s = collision_system(nb, 1025)
    T = 2 + len(s.devices)
    before = nb.kernel_launches()
    evs, _, pairs = nb.solve_partial(s, 0, 1, T, n_steps=20000, all_devices=True)
    launches = nb.kernel_launches() - before
    assert evs[1].hit_step == evs[1].steps_done == 476
    assert pairs == 476 * s.n * (s.n - 1)
    assert 3 * 476 < launches <= 3 + 3 * (476 + 2 * MAX_CHUNK)


def test_two_gpus(nb, kats):
    if nb.device_count() < 2:
        pytest.skip("needs two GPUs")
    s = padded(nb, "b20", 1025)
    one = nb.solve(s, gpus=[0])
    two = nb.solve(s, gpus=2)
    assert fields(two) == fields(one)
    check_golden(two, "b20", kats)
