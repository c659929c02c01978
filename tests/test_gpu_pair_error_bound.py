"""The FAST pair term of every kernel path against an extended-precision reference, to a few ulp.

DESIGN §3 states that the FAST pair term (rsqrt seed, e = 1 - r2*y0^2, p = 1 + 1.5e + 1.875e^2) has a truncation
below 2^-55 on top of a handful of roundings.  The FAST-tolerance tests elsewhere (q within 2 ulp, v within 1e-12)
cannot see an error of a few thousand ulp, which is what a wrong second-order coefficient gives; these tests can.

Sparse-source systems: only k <= 16 bodies (the sources) have mass.  A massless body adds exactly 0 in every FAST form
(c = 0 and fma(0, d, a) = a; the self term is +0), so the acceleration of every body is a sum of at most k pair terms
and a bound of a few ulp holds at any n.  One step from rest gives v1 = round(a*dt), and every component must satisfy

    |v1 - dt*a_exact| <= (K + k) * u * dt * sum_j |term_ij|,    u = 2^-53,

with K = 8 counted from the operations of one term (dx, the r2 chain, the seed correction with its truncation
<= 2.2|e|^3, five products, the accumulate and the product with dt) and k for the order of the accumulation.
The reference is the exact sum on the kernel's double inputs, evaluated in long double (checked against mpmath).

Which kernel runs (launch_traj_batch in nb_traj.cu, DeviceBatch::run and run_steps_large in nb_host.cu):
  * nb_run_steps and Trajectory take the whole-GPU grid kernel for 128 <= n <= 1024 when the device supports it, so
    the single-block kernels are reached through ensemble_run, which never takes the grid kernel;
  * traj_kernel<FAST, JS> with JS > 1 for n <= 512, traj_kernel<FAST, 1> for 512 < n <= 896, traj_sym_kernel for
    896 < n <= 1024;
  * n > 1024: run_steps takes the symmetric stepper (sym_accel_kernel<6> or <8> by shard size), ShardedSystem the row
    kernel large_accel_kernel<FAST>.
test_each_case_runs_the_kernel_it_names checks this routing with the CUDA profiler."""
import math

import numpy as np
import pytest

U = 2.0 ** -53
K = 8
DT = 60.0
G = 6.674e-11
EPS2 = 1e-3 * 1e-3  # the kernels' EPS * EPS, the same double


def fst(step):
    """|sin(step*dt/6000)|: the host table's formula (nb_host.cu), through the same libm sin."""
    return abs(math.sin((step * 60.0) / 6000))


def gm_of(m, is_device, step):
    """G*m_eff of every body at `step`, rounded in double exactly as gm_eff (nb_math.cuh) rounds it."""
    m = np.asarray(m, dtype=np.float64)
    return np.where(np.asarray(is_device) != 0, G * (m + (0.5 * m) * fst(step)), G * m)


def exact_accel(q, gm, dt):
    """dt * sum_j gm_j d_ij / (|d_ij|^2 + eps^2)^(3/2) and dt * sum_j |term_ij| per component, both [3, n] long double,
    on the kernel's double inputs (planar q[3n], gm[n]).  Massless bodies contribute exactly 0 and are skipped."""
    assert np.finfo(np.longdouble).nmant >= 63, "the reference needs an extended long double"
    n = len(gm)
    x = np.asarray(q, dtype=np.float64).reshape(3, n).astype(np.longdouble)
    a = np.zeros((3, n), dtype=np.longdouble)
    s = np.zeros((3, n), dtype=np.longdouble)
    for j in np.nonzero(gm)[0]:
        d = x[:, j:j + 1] - x
        r2 = (d[0] * d[0] + d[1] * d[1]) + d[2] * d[2] + np.longdouble(EPS2)
        t = np.longdouble(gm[j]) * d / (r2 * np.sqrt(r2))
        a += t
        s += np.abs(t)
    return a * np.longdouble(dt), s * np.longdouble(dt)


def source_terms(q, gm, i, c):
    """|term_ij| of body i, component c, for every source j: the source that dominates a failing body."""
    n = len(gm)
    x = np.asarray(q).reshape(3, n).astype(np.longdouble)
    best, arg = np.longdouble(-1), -1
    for j in np.nonzero(gm)[0]:
        d = x[:, j] - x[:, i]
        r2 = d @ d + np.longdouble(EPS2)
        t = abs(np.longdouble(gm[j]) * d[c] / (r2 * np.sqrt(r2)))
        if t > best:
            best, arg = t, int(j)
    return arg


def check_bound(v1, q, gm, label, per_pair=False):
    """v1 (planar [3n]) after one step from rest against the exact dt*a; returns the largest error in units of
    u * dt * sum_j |term_ij|.  per_pair: every body has one term at most, bound K*u."""
    n = len(gm)
    k = int(np.count_nonzero(gm))
    ref, scale = exact_accel(q, gm, DT)
    err = np.abs(np.asarray(v1, dtype=np.float64).reshape(3, n).astype(np.longdouble) - ref)
    allow = K if per_pair else K + k
    bad = err > allow * U * scale
    with np.errstate(divide="ignore", invalid="ignore"):
        ulp = np.where(scale > 0, err / (U * scale), np.where(err > 0, np.inf, 0.0))
    worst = float(ulp.max())
    c, i = np.unravel_index(int(np.argmax(ulp)), ulp.shape)
    print("pair error bound, %s: max %.3f u (bound %d u)" % (label, worst, allow))
    assert not bad.any(), ("%s: %d components over the bound; worst body %d, component %d, worst source %d: %.2f u "
                           "(bound %d u, v1 %r, exact %r)" % (label, int(bad.sum()), i, c, source_terms(q, gm, i, c), worst,
                                                            allow, float(np.asarray(v1).reshape(3, n)[c, i]),
                                                            float(ref[c, i])))
    return worst


# ---- geometry ----------------------------------------------------------------------------------------------------
def _unit(rng, count):
    d = rng.normal(size=(count, 3))
    return d / np.linalg.norm(d, axis=1, keepdims=True)


def axis_distance(t):
    """d with fl(d*d + eps^2) ~ t: a probe at (d, 0, 0) from a source at the origin has r2 ~ t."""
    return math.sqrt(max(t - EPS2, 0.0))


# r2 targets for probes on the x axis of the source at the origin: both exponent parities (the seed works on r2 scaled
# into [1, 4) by an even power of two) with mantissas next to 1, 2 and 4
SPECIAL_R2 = [4.0 ** E * f for E in (-9, -1, 0, 6, 21, 50)
              for f in (1.0, 1.0 + 2.0 ** -40, 2.0 * (1 - 2.0 ** -40), 2.0, 2.0 * (1 + 2.0 ** -40), 4.0 * (1 - 2.0 ** -40))]


def sparse_system(nb, n, sources, seed, device=True):
    """n bodies at rest; the bodies `sources` have mass (one of them a gravity device), the others are massless probes.
    Source sources[0] sits at the origin; the others within 1e8 m of it.  The first probes are: one coincident with
    the origin source, one 3e-4 m from it (closer than eps), then probes on the x axis at the SPECIAL_R2 targets; the
    rest are placed 1e-4 .. 1e15 m from a random source in a random direction.  Planet and asteroid are two probes
    2e13 m apart (no hit at step 0).  Masses are log-uniform, G*m from ~7e-11 to ~7e20; the device is heavy."""
    rng = np.random.default_rng(seed)
    sources = sorted(set(int(j) for j in sources))
    assert len(sources) <= 16 and sources[-1] < n
    x = np.zeros((n, 3))
    for j, r, u in zip(sources[1:], 10.0 ** rng.uniform(-2, 8, len(sources) - 1), _unit(rng, len(sources) - 1)):
        x[j] = r * u
    src0 = sources[0]
    probes = [i for i in range(n) if i not in set(sources)]
    special = [np.zeros(3), np.array([3e-4, 0.0, 0.0])] + [np.array([axis_distance(t), 0.0, 0.0]) for t in SPECIAL_R2]
    planet = asteroid = 0
    if len(probes) >= 3:
        planet, asteroid = probes.pop(), probes.pop()
        x[planet] = (1e13, 0.0, 0.0)
        x[asteroid] = (-1e13, 0.0, 0.0)
    for i, p in zip(probes, special):
        x[i] = x[src0] + p
    rest = probes[len(special):]
    hosts = rng.choice(sources, size=len(rest))
    for i, h, r, u in zip(rest, hosts, 10.0 ** rng.uniform(-4, 15, len(rest)), _unit(rng, len(rest))):
        x[i] = x[h] + r * u
    m = np.zeros(n)
    m[sources] = 10.0 ** rng.uniform(0, 31, len(sources))  # G*m from ~7e-11 to ~7e20
    dev = np.zeros(n, dtype=np.uint8)
    if device:
        j = sources[len(sources) // 2]
        dev[j] = 1
        m[j] = 10.0 ** rng.uniform(29, 31)  # heavy, so that its mass modulation shows on the probes around it
    q = np.ascontiguousarray(x.T).reshape(-1)
    return nb.System(n, planet, asteroid, q, np.zeros(3 * n), m, dev)


def sweep_probes(count=4096, seed=1):
    """Probe offsets from a source at the origin with r2 sweeping 2^-20 .. 2^120 (r2 >= eps^2 ~ 2^-19.93): 29 mantissas in
    each of the 140 binades, random directions; the remaining probes at random r2 in the range."""
    rng = np.random.default_rng(seed)
    t = [2.0 ** b * f for b in range(-20, 120) for f in np.linspace(1.0, 2.0, 29, endpoint=False)]
    t += list(2.0 ** rng.uniform(-20, 120, count - len(t)))
    d = np.array([math.sqrt(max(ti - EPS2, 0.0)) for ti in t])
    return d[:, None] * _unit(rng, count)


def with_source_at_origin(nb, offsets, gm_source=6.674e9):
    n = len(offsets) + 1
    x = np.zeros((n, 3))
    x[1:] = offsets
    m = np.zeros(n)
    m[0] = gm_source / G
    return nb.System(n, 0, 0, np.ascontiguousarray(x.T).reshape(-1), np.zeros(3 * n), m, np.zeros(n, dtype=np.uint8))


# ---- the CPU check of the reference --------------------------------------------------------------------------------
def test_exact_accel_matches_mpmath():
    """The long-double reference against mpmath at 50 digits, term by term (one source, massless probes): coincident
    bodies, separations far below eps, 1e15 m, and random separations from 1e-4 to 1e15 m."""
    import mpmath

    rng = np.random.default_rng(3)
    src = np.array([1234.5678, -9.87654321e5, 3.3e-2])
    offs = [np.zeros(3), np.array([1e-9, 0, 0]), np.array([2e-5, -3e-5, 1e-5]), np.array([3e-4, 0, 0]),
            np.array([1e15, 0, 0]), np.array([-6e14, 7e14, 2e14])]
    offs += list(10.0 ** rng.uniform(-4, 15, 300)[:, None] * _unit(rng, 300))
    n = len(offs) + 1
    x = np.zeros((n, 3))
    x[0] = src
    x[1:] = src + np.array(offs)
    q = np.ascontiguousarray(x.T).reshape(-1)
    for gm0 in (6.674e-11, 3.7e20):
        gm = np.zeros(n)
        gm[0] = gm0
        a, s = exact_accel(q, gm, 1.0)
        assert np.array_equal(np.abs(a), s)  # one term per probe
        mpmath.mp.dps = 50
        e2 = mpmath.mpf(EPS2)
        worst = 0.0
        for i in range(1, n):
            d = [mpmath.mpf(float(x[0, c])) - mpmath.mpf(float(x[i, c])) for c in range(3)]
            r2 = d[0] ** 2 + d[1] ** 2 + d[2] ** 2 + e2
            inv = mpmath.mpf(gm0) / (r2 * mpmath.sqrt(r2))
            for c in range(3):
                t = d[c] * inv
                err = abs(_ld_to_mpf(a[c, i]) - t)
                assert err <= mpmath.mpf(2) ** -60 * abs(t), (i, c, float(err / abs(t)) if t else float(err))
                if t:
                    worst = max(worst, float(err / abs(t)))
        assert worst < 2.0 ** -60


def _ld_to_mpf(v):
    """A long double as an exact mpmath number: mantissa and exponent through frexp (64-bit mantissa, exact)."""
    import mpmath

    mant, ex = np.frexp(v)
    mi = int(np.ldexp(mant, 64))  # exact: the mantissa has at most 64 bits
    return mpmath.mpf(mi) * mpmath.mpf(2) ** (int(ex) - 64)


def test_gm_of_is_the_kernels_mass_rule():
    """The host twin of the device mass: G*(m0 + (0.5*m0)*fst) for devices, G*m0 for the other bodies."""
    m = np.array([1.0, 3.3e30, 7.0e21])
    dev = np.array([0, 1, 1], dtype=np.uint8)
    g = gm_of(m, dev, 101)
    assert g[0] == G * 1.0
    assert g[1] == G * (3.3e30 + (0.5 * 3.3e30) * abs(math.sin(101 * 60.0 / 6000)))
    assert gm_of(m, dev, 0)[2] == G * 7.0e21


# ---- GPU: one case per kernel path and tiling edge ----------------------------------------------------------------
# (path, n, sources).  Sources sit on the edges of what the kernel tiles: JS slices, 128-body groups and their
# 64-body halves (traj_sym_kernel), rows and their diagonal (sym_accel_kernel: stride = nb_sym_row_stride), shard
# boundaries (multi-rank), j splits and the partial last 256-record tile (large_accel_kernel).
SMALL = [
    ("traj_js", 2, [0]),
    ("traj_js", 33, [0, 15, 16, 32]),
    ("traj_js", 300, [0, 1, 150, 298, 299]),
    ("traj_js", 512, [0, 255, 256, 510, 511]),
    ("traj_1", 700, [0, 349, 350, 699]),
    ("traj_1", 896, [0, 447, 448, 895]),
    ("traj_sym", 897, [0, 63, 64, 127, 128, 511, 512, 575, 576, 895, 896]),
    ("traj_sym", 1000, [0, 127, 128, 383, 384, 575, 576, 639, 640, 895, 896, 960, 999]),
    ("traj_sym", 1024, [0, 63, 64, 127, 128, 255, 256, 511, 512, 575, 576, 767, 768, 895, 896, 1023]),
    ("grid", 256, [0, 1, 127, 128, 253]),
    ("grid", 1000, [0, 511, 512, 996, 997]),
    ("grid", 1024, [0, 127, 128, 1020, 1021]),
]
LARGE = [
    # sym_accel_kernel<6>: 1025 / 1536 are one diagonal row; 2049 = rows [0, 1025) and [1025, 2049)
    ("sym_accel", 1025, [0, 31, 32, 512, 1023, 1024]),
    ("sym_accel", 1536, [0, 127, 128, 767, 768, 1535]),
    ("sym_accel", 2049, [0, 500, 1023, 1024, 1025, 1026, 1152, 1153, 2047, 2048]),
    # sym_accel_kernel<8>: rows [0, 2048) / [2048, 4096) and [0, 1667) / [1667, 3333)
    ("sym_accel", 4096, [0, 1000, 2047, 2048, 2049, 2175, 2176, 4094, 4095]),
    ("sym_accel", 3333, [0, 800, 1666, 1667, 1668, 1794, 1795, 3331, 3332]),
    # row kernel: 1025 = splits [0, 768) / [768, 1025); 4196 = 6 splits of 768, last tile [4096, 4196)
    ("large_accel", 1025, [0, 255, 256, 767, 768, 1023, 1024]),
    ("large_accel", 4196, [0, 767, 768, 3839, 3840, 4095, 4096, 4150, 4195]),
]
MULTI = [
    (6144, 2, [0, 1535, 1536, 3071, 3072, 3073, 4607, 4608, 6143]),
    (6144, 3, [0, 1000, 2047, 2048, 4095, 4096, 5000, 6143]),
    (8192, 8, [0, 1023, 1024, 2047, 2048, 3071, 3072, 4095, 4096, 5119, 5120, 6143, 6144, 7167, 7168, 8191]),
]
KERNEL = {"traj_js": "traj_kernel<0,%d>(", "traj_1": "traj_kernel<0,1>(", "traj_sym": "traj_sym_kernel(",
          "grid": "grid_traj_kernel<1,false>(", "sym_accel": "sym_accel_kernel<%d>(", "large_accel": "large_accel_kernel<0>("}


def _ids(cases):
    return ["%s-%d" % (c[0], c[1]) for c in cases]


def run_small(nb, path, systems):
    """One step from rest of each system on the kernel `path` names; returns v [S, 3n]."""
    if path == "grid":
        out = []
        for s in systems:
            t = nb.Trajectory(s, nb.KIND_Q2)
            ev = t.run(1)
            q, v, m, step = t.state()
            t.close()
            assert step == 1 and ev.steps_done == 1 and ev.hit_step == -2
            out.append(v)
        return np.stack(out)
    q = np.stack([s.q for s in systems])
    v = np.zeros_like(q)
    m = np.stack([s.m for s in systems])
    dev = np.stack([s.is_device for s in systems])
    ev, _ = nb.ensemble_run(q, v, m, dev, [s.planet for s in systems], [s.asteroid for s in systems], kind=nb.KIND_PLAIN,
                            step_end=1)
    assert all(e.steps_done == 1 for e in ev)
    return v


def run_large(nb, path, s):
    if path == "large_accel":
        import torch

        sh = nb.ShardedSystem(s, 0, 1, device="cuda:0")
        sh.advance(1)
        torch.cuda.synchronize()
        return sh.velocities()
    q, v = s.q.copy(), s.v.copy()
    nb.run_steps(0, 1, s.n, q, v, s.m, s.is_device)
    return v


def run_multi(nb, s, world):
    w = nb.SymLocalWorld(s, world, device="cuda:0")
    w.advance(1)
    w.positions()  # raises if a rank's wait timed out
    v = w.velocities()
    w.close()
    return v


@pytest.mark.gpu
@pytest.mark.parametrize("path,n,sources", SMALL, ids=_ids(SMALL))
def test_sparse_sources_small_paths(nb, path, n, sources):
    """Single-block kernels (two systems in one launch: the second has its sources mirrored) and the grid kernel."""
    mirrored = [n - 1 - j for j in sources]
    systems = [sparse_system(nb, n, sources, seed=n), sparse_system(nb, n, mirrored, seed=n + 1)]
    v = run_small(nb, path, systems)
    for k, s in enumerate(systems):
        check_bound(v[k], s.q, gm_of(s.m, s.is_device, 1), "%s n=%d system %d" % (path, n, k))


@pytest.mark.gpu
@pytest.mark.parametrize("path,n,sources", LARGE, ids=_ids(LARGE))
def test_sparse_sources_large_paths(nb, path, n, sources):
    s = sparse_system(nb, n, sources, seed=n)
    v = run_large(nb, path, s)
    check_bound(v, s.q, gm_of(s.m, s.is_device, 1), "%s n=%d" % (path, n))


@pytest.mark.gpu
@pytest.mark.parametrize("n,world,sources", MULTI, ids=["%d-%d" % c[:2] for c in MULTI])
def test_sparse_sources_multi_rank_symmetric(nb, n, world, sources):
    """Partial rows PJ stored into the owner rank: sources on both sides of every shard boundary."""
    s = sparse_system(nb, n, sources, seed=n + world)
    v = run_multi(nb, s, world)
    check_bound(v, s.q, gm_of(s.m, s.is_device, 1), "multi-rank n=%d world=%d" % (n, world))


@pytest.mark.gpu
def test_each_case_runs_the_kernel_it_names(nb):
    """The routing the cases above rely on, from the CUDA profiler's kernel records (one system per case)."""
    from torch.profiler import ProfilerActivity, profile

    def launched(fn):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
        return {e.name.replace(" ", "") for e in prof.events()}

    for path, n, sources in SMALL + LARGE:
        s = sparse_system(nb, n, sources, seed=n)
        want = KERNEL[path]
        if path == "sym_accel":
            want %= 8 if n in (3333, 4096) else 6
        elif path == "traj_js":
            want %= {2: 32, 33: 16, 300: 2, 512: 2}[n]
        small = (path, n, sources) in SMALL
        names = launched(lambda: run_small(nb, path, [s]) if small else run_large(nb, path, s))
        assert any(want in x for x in names), (path, n, want, sorted(names))
    for n, world, ipl in ((6144, 2, 6), (6144, 3, 8), (8192, 8, 6)):
        s = sparse_system(nb, n, [0, n - 1], seed=1)
        names = launched(lambda: run_multi(nb, s, world))
        assert any(("sym_accel_kernel<%d>(" % ipl) in x for x in names), (n, world, sorted(names))


# ---- GPU: the seed's accuracy, measured ---------------------------------------------------------------------------
@pytest.mark.gpu
def test_seed_sweep_one_pair_per_probe(nb):
    """One source at the origin, 4096 massless probes with r2 from eps^2 to 2^120, several mantissas per binade: each
    probe's velocity is one pair term, bounded by K*u.  n > 1024 (the symmetric stepper's one-sided diagonal and, on the
    source's side, pair_sym) and n = 512 (traj_kernel<FAST, 2>, eight systems of 511 probes in one launch)."""
    offs = sweep_probes()
    s = with_source_at_origin(nb, offs)
    q, v = s.q.copy(), s.v.copy()
    nb.run_steps(0, 1, s.n, q, v, s.m, s.is_device)
    worst = [check_bound(v, s.q, gm_of(s.m, s.is_device, 1), "seed sweep, n=%d" % s.n, per_pair=True)]
    systems = [with_source_at_origin(nb, offs[k * 511:(k + 1) * 511]) for k in range(8)]
    v = run_small(nb, "traj_js", systems)
    for k, sk in enumerate(systems):
        worst.append(check_bound(v[k], sk.q, gm_of(sk.m, sk.is_device, 1), "seed sweep, n=512 system %d" % k, per_pair=True))
    print("seed sweep: max %.3f u over %d pair terms" % (max(worst), 2 * len(offs)))


# ---- GPU: the large path resumed at a later step -------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n", [1025, 2049])
def test_large_path_resumed_step_device_mass(nb, oracle, n):
    """run_steps(100, 101) packs the first step's records with the device masses of step 101: STRICT bit-identical to
    the oracle, FAST within the sparse bound of the exact accelerations at fst[101]."""
    sources = [0, n // 2, n - 1]
    s = sparse_system(nb, n, sources, seed=7 * n)
    assert s.is_device[n // 2]
    q, v = s.q.copy(), s.v.copy()
    nb.run_steps(100, 101, n, q, v, s.m, s.is_device, math=nb.MATH_STRICT)
    qo, vo = s.q.copy(), s.v.copy()
    oracle.run_steps(oracle.MODE_SQRT3, n, qo, vo, s.m, s.is_device, 100, 101)
    assert np.array_equal(q, qo) and np.array_equal(v, vo)
    q, v = s.q.copy(), s.v.copy()
    nb.run_steps(100, 101, n, q, v, s.m, s.is_device)
    check_bound(v, s.q, gm_of(s.m, s.is_device, 101), "resumed at step 100, n=%d" % n)
