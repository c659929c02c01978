"""GPU: the diagnostics (nb_diagnostics, nb_traj_diagnostics) against the long-double reference, batch and handle identities,
and the conservation of momentum and angular momentum over 1 000 steps.

Error bound of one quantity (csrc/nb_diag.cu, DESIGN.md §4.6), |gpu - exact| <= (c + L + D) * u * scale, u = 2^-53.
scale is the value itself for mass, kinetic and potential (their terms all have one sign), and sum |terms| per component
for momentum (terms m_i v_i) and angular momentum (terms m_i q_a v_b and m_i q_b v_a, the two products of a component).

c, the roundings of one term:
  potential  10: dx, dy, dz and the three FMAs of r2 (<= 5u on r2, eps^2 rounded to double 0.5u, halved by the square
                 root: 2.75u), y0^2 (0.5u), the last FMA of r^-1 (1u), the seed's truncation (< 0.25u), the two effective
                 masses rounded to double (2u each), the final product with G (1u);
  mass        2: m0 + (0.5 m0)|sin| rounded twice (devices);
  kinetic     5: vz^2 and two FMAs (3u), the effective mass (2u); the product with m is inside the accumulating FMA, 0.5 exact;
  momentum    2: the effective mass; the product with m is inside the accumulating FMA;
  ang. mom.   4: fma(y, vz, -(z*vy)) <= 2u of |y vz| + |z vy|, the effective mass (2u).
L, the longest serial chain: a thread adds one tile of T = 256 j terms per i body (potential), then its IPT = 4 i bodies;
  the O(n) terms are a chain of the IPT = 4 bodies.  So L = T + IPT = 260 for the potential and 4 for the others.
D, the tree depth: 6 levels over the 64 threads of a tile block (5 shuffle levels + 2 warps), then per system each of
  the 1 024 threads of the sum kernel adds every 1 024-th tile partial (a chain of ceil(K / 1024) for K tiles), then 10
  levels (5 shuffle levels + 32 warps).  D = 16 + ceil(K / 1024); K = t(t+1)/2, t = ceil(n / 256).
At 65 536 bodies K = 32 896 and the potential's bound is (10 + 260 + 49) u = 3.5e-14.  The reference, diag_reference
(tests/diag_reference.cc: long double, compensated sums), is within 2^-60 of sum |terms| (test_diag_cpu.py)."""
import math

import numpy as np
import pytest
from conftest import CASES, case_path

import diag_reference

pytestmark = pytest.mark.gpu

U = 2.0 ** -53
T, IPT = 256, 4
G = 6.674e-11
DT = 60.0
C_TERM = dict(mass=2, kinetic=5, potential=10, momentum=2, angular_momentum=4)
WORST = {}


def depth(n):
    t = -(-n // T)
    return 16 + -(-(t * (t + 1) // 2) // 1024)


def bound_units(key, n):
    return C_TERM[key] + (T + IPT if key == "potential" else IPT) + depth(n)


def fst(step):
    return abs(math.sin((step * 60.0) / 6000))


def m_eff(m, dev, step):
    m = np.asarray(m, dtype=np.float64)
    return np.where(np.asarray(dev) != 0, m + (0.5 * m) * fst(step), m)


def scales(n, q, v, me):
    """sum |terms| per component of momentum and angular momentum (float64 suffices for a bound's scale)."""
    x, u = q.reshape(3, n), v.reshape(3, n)
    p = np.abs(me * u).sum(axis=1)
    lm = np.array([(np.abs(me * x[(c + 1) % 3] * u[(c + 2) % 3]) + np.abs(me * x[(c + 2) % 3] * u[(c + 1) % 3])).sum()
                   for c in range(3)])
    return p, lm


def check(got, ref, n, q, v, me, label):
    """Every quantity of `got` (nb_diag dict) within its bound of `ref` (reference dict); records the largest error in u."""
    p_scale, l_scale = scales(n, q, v, me)
    for key in ("mass", "kinetic", "potential", "momentum", "angular_momentum"):
        g = np.atleast_1d(np.asarray(got[key], dtype=np.float64)).astype(np.longdouble)
        r = np.atleast_1d(ref[key])
        sc = {"momentum": p_scale, "angular_momentum": l_scale}.get(key, np.abs(r.astype(np.float64)))
        err = np.abs(g - r).astype(np.float64)
        with np.errstate(divide="ignore", invalid="ignore"):
            units = np.where(sc > 0, err / (U * sc), np.where(err > 0, np.inf, 0.0))
        lim = bound_units(key, n)
        WORST[key] = max(WORST.get(key, 0.0), float(units.max()))
        print("%s %s: %.3f u (bound %d u)" % (label, key, float(units.max()), lim))
        assert (units <= lim).all(), (label, key, units.tolist(), lim)


def check_system(nb, s, step, label):
    got = nb.diagnostics(s.q, s.v, s.m, s.is_device, step=step)
    assert got["n"] == s.n and got["step"] == step
    ref = diag_reference.diagnostics(s.n, s.q, s.v, s.m, s.is_device, step)
    check(got, ref, s.n, s.q, s.v, m_eff(s.m, s.is_device, step), label)
    return got


def one_body(nb):
    return nb.System(1, 0, 0, np.array([1e11, -2e11, 3e10]), np.array([4e3, 5e3, -6e3]), np.array([7e29]),
                     np.ones(1, np.uint8))


SIZES = [1, 2, 3, T - 1, T, T + 1, 1000, 1024, 1025, 4096, 65536]


@pytest.mark.parametrize("n", SIZES)
def test_accuracy_against_reference(nb, n):
    s = one_body(nb) if n == 1 else nb.generate_system(n, seed=n, n_devices=min(4, n - 2))
    check_system(nb, s, 0, "n=%d" % n)
    if n == 65536:
        print("bound at 65536 bodies: potential %.3g" % (bound_units("potential", n) * U))
        assert bound_units("potential", n) * U <= 1e-13


@pytest.mark.parametrize("case", CASES)
def test_accuracy_goldens(nb, case):
    check_system(nb, nb.read_input(case_path(case)), 0, case)


def test_accuracy_modulated_devices(nb):
    s = nb.generate_system(3000, seed=5, n_devices=64)
    assert fst(12345) > 0.1
    got = check_system(nb, s, 12345, "synthetic 3000 bodies, 64 devices, step 12345")
    assert got != nb.diagnostics(s.q, s.v, s.m, s.is_device, step=0)  # the modulation shows


def test_report_worst_error():
    """Runs after the accuracy tests of this module: the largest error seen, in units of u."""
    print("diagnostics, largest error in u: " + ", ".join("%s %.3f" % kv for kv in sorted(WORST.items())))


# ---- batches -----------------------------------------------------------------------------------------------------
def test_batch_equals_single_bit_for_bit(nb):
    n, S = 700, 7
    systems = [nb.generate_system(n, seed=100 + k, n_devices=[0, 1, 4, 13, 64, 2, 0][k]) for k in range(S)]
    for k, s in enumerate(systems):
        s.v *= 1.0 + k
    q, v = np.stack([s.q for s in systems]), np.stack([s.v for s in systems])
    m, dev = np.stack([s.m for s in systems]), np.stack([s.is_device for s in systems])
    batch = nb.diagnostics(q, v, m, dev, step=4321)
    assert batch == nb.diagnostics(q, v, m, dev, step=4321)  # identical calls, identical bits
    for k, s in enumerate(systems):
        assert batch[k] == nb.diagnostics(s.q, s.v, s.m, s.is_device, step=4321), k


def test_c4_shape_1024_by_1024(nb):
    """Config C4: 1 024 members of one 1 024-body system, velocities scaled by (1 + 1e-9 k)."""
    base = nb.generate_system(1024, seed=42)
    S = 1024
    q = np.tile(base.q, (S, 1))
    v = np.stack([base.v * (1.0 + 1e-9 * k) for k in range(S)])
    m, dev = np.tile(base.m, (S, 1)), np.tile(base.is_device, (S, 1))
    batch, secs = nb.diagnostics(q, v, m, dev, step=77, return_seconds=True)
    print("C4 shape: %.3f ms of kernels" % (secs * 1e3))
    for k in (0, 1, 511, 1023):
        ref = diag_reference.diagnostics(1024, q[k], v[k], m[k], dev[k], 77)
        check(batch[k], ref, 1024, q[k], v[k], m_eff(m[k], dev[k], 77), "C4 member %d" % k)
        assert batch[k] == nb.diagnostics(q[k], v[k], m[k], dev[k], step=77)


# ---- trajectory handles ------------------------------------------------------------------------------------------
def handle_matches_state(nb, t, is_device, gpu=0):
    """t.diagnostics() == nb_diagnostics of nb_traj_state's q, v, m at its step, bit for bit."""
    got = t.diagnostics()
    q, v, m, step = t.state()
    assert got["step"] == step
    assert got == nb.diagnostics(q, v, m, is_device, step=step, gpu=gpu)
    return got, m, step


def test_handles_equal_state_diagnostics(nb):
    from test_gpu_large_queries import collision_system

    s = collision_system(nb, 512)
    heavy = 3
    assert s.is_device[heavy]
    t1 = nb.Trajectory(s, nb.KIND_Q1)
    t1.run(300)
    got, m, step = handle_matches_state(nb, t1, s.is_device)
    assert step == 300 and np.all(m[s.is_device != 0] == 0)  # Q1: devices massless
    t2 = nb.Trajectory(s, nb.KIND_Q2)
    ev = t2.run(1000)
    assert ev.hit_step != -2
    got, m, step = handle_matches_state(nb, t2, s.is_device)
    assert step == ev.hit_step  # stopped at its hit
    t3 = nb.Trajectory(s, nb.KIND_Q3, destroy_device=heavy)
    ev = t3.run(400)
    assert ev.destroyed_step != -2
    got, m, step = handle_matches_state(nb, t3, s.is_device)
    assert step > ev.destroyed_step and m[heavy] == 0  # after its destroy step, mass zeroed
    if nb.device_count() >= 2:
        f = t1.fork(nb.KIND_Q1, gpu=1)
        got_f, _, step_f = handle_matches_state(nb, f, s.is_device, gpu=1)
        assert step_f == 300 and got_f == t1.diagnostics()
        f.close()
    for t in (t1, t2, t3):
        t.close()


# ---- conservation, no reference ----------------------------------------------------------------------------------
K_PAIR = 8  # roundings of one FAST pair term, dt product included (test_gpu_pair_error_bound.py)


def step_bounds(n, q, m, q1, v1):
    """First-order bounds on the change of exact P and L over one step (q, v) -> (q1, v1), from the roundings of the step.
    The kick gives v1 = v + a dt + eps with |eps_ic| <= (K_PAIR + n) u S_ic + u |v1_ic|, where S_ic = dt sum_j |term_ij|
    (K_PAIR per pair term, n for any order of the accumulation); the drift q1 = q + v1 dt + e3 with
    |e3_ic| <= u (|v1_ic| dt + |q1_ic|).  Exact arithmetic conserves both (sum m a = 0, sum m q x a = 0 for central pair
    forces), so  |dP_c| <= sum_i m_i eps_ic  and
    |dL_x| <= sum_i m_i (|y_i| eps_iz + |z_i| eps_iy + e3_iy |v1_iz| + e3_iz |v1_iy|)  (cyclically)."""
    import torch

    dv = torch.device("cuda:0")
    x = torch.tensor(q.reshape(3, n).T.copy(), dtype=torch.float64, device=dv)
    gm = torch.tensor(G * m, dtype=torch.float64, device=dv)
    d = x[None, :, :] - x[:, None, :]  # d[i, j] = x_j - x_i
    r2 = (d * d).sum(-1) + 1e-6
    w = gm[None, :] / (r2 * torch.sqrt(r2))
    S = DT * (w[:, :, None] * d.abs()).sum(1).cpu().numpy().T  # [3, n]
    v1p, q1p, qp = v1.reshape(3, n), q1.reshape(3, n), q.reshape(3, n)
    eps = (K_PAIR + n) * U * S + U * np.abs(v1p)
    e3 = U * (np.abs(v1p) * DT + np.abs(q1p))
    dp = (m * eps).sum(axis=1)
    dl = np.array([(m * (np.abs(qp[(c + 1) % 3]) * eps[(c + 2) % 3] + np.abs(qp[(c + 2) % 3]) * eps[(c + 1) % 3]
                         + e3[(c + 1) % 3] * np.abs(v1p[(c + 2) % 3]) + e3[(c + 2) % 3] * np.abs(v1p[(c + 1) % 3]))).sum()
                   for c in range(3)])
    return dp, dl


def diag_error(n, q, v, m, key):
    p_scale, l_scale = scales(n, q, v, m)
    return bound_units(key, n) * U * (p_scale if key == "momentum" else l_scale)


@pytest.mark.parametrize("n", [1024, 2048], ids=["grid-kernel-1024", "symmetric-stepper-2048"])
def test_momentum_and_angular_momentum_conserved(nb, n):
    """1 000 steps of a device-free synthetic system through nb_run_steps, one call per step (n = 2048 takes the symmetric
    large-N stepper); |P_1000 - P_0| and |L_1000 - L_0| within the summed per-step bounds plus the diagnostics' own
    bound at both ends."""
    s = nb.generate_system(n, seed=2024, n_devices=0)
    assert not s.is_device.any()
    q, v = s.q.copy(), s.v.copy()
    d0 = nb.diagnostics(q, v, s.m, s.is_device, step=0)
    allow_p = diag_error(n, q, v, s.m, "momentum")
    allow_l = diag_error(n, q, v, s.m, "angular_momentum")
    for step in range(1, 1001):
        q0 = q.copy()
        nb.run_steps(step - 1, step, n, q, v, s.m, s.is_device)
        dp, dl = step_bounds(n, q0, s.m, q, v)
        allow_p += dp
        allow_l += dl
    d1 = nb.diagnostics(q, v, s.m, s.is_device, step=1000)
    allow_p += diag_error(n, q, v, s.m, "momentum")
    allow_l += diag_error(n, q, v, s.m, "angular_momentum")
    dP = np.abs(np.array(d1["momentum"]) - np.array(d0["momentum"]))
    dL = np.abs(np.array(d1["angular_momentum"]) - np.array(d0["angular_momentum"]))
    e0, e1 = d0["energy"], d1["energy"]
    print("n=%d: |dP| / bound %s, |dL| / bound %s, relative energy drift %.3e" % (n, (dP / allow_p).round(4).tolist(),
                                                                                 (dL / allow_l).round(4).tolist(),
                                                                                 (e1 - e0) / abs(e0)))
    assert (dP <= allow_p).all(), (dP, allow_p)
    assert (dL <= allow_l).all(), (dL, allow_l)
