"""CPU: the diagnostics (nb_diagnostics, nb_traj_diagnostics) without a GPU.

  * diag_reference (tests/diag_reference.cc), the long-double reference of tests/test_gpu_diagnostics.py, against
    mpmath at 50 digits: every quantity within 2^-60 of sum |terms| on crafted systems (coincident bodies, 1e30 kg
    beside massless bodies, coordinates near 2e20 m as in the goldens, gravity devices at a step where |sin| != 0);
  * the nb_diag layout of include/nbody_b200.h against the ctypes mirror;
  * argument validation (NB_ERR_ARG before any GPU check) and NB_ERR_NO_GPU without a device;
  * `nbtool diag` without a file prints the usage;
  * the kernels are in the built library, with MUFU.RSQ64H and DFMA and no atomics, and ptxas reports no spills."""
import ctypes as C
import math
import os
import re
import shutil
import subprocess

import numpy as np
import pytest
from conftest import ROOT

import diag_reference

G = 6.674e-11
EPS = 1e-3


def fst(step):
    return abs(math.sin((step * 60.0) / 6000))


def exact_terms(n, q, v, m, dev, step):
    """(value, sum |terms|) of every quantity in mpmath at 50 digits, the definitions of include/nbody_b200.h on the double
    inputs; m_eff = m0 + 0.5*m0*|sin| with the double |sin| the library uses."""
    import mpmath

    mpmath.mp.dps = 50
    f = mpmath.mpf(fst(step))
    me = [mpmath.mpf(float(m[i])) * (1 + f / 2) if dev[i] else mpmath.mpf(float(m[i])) for i in range(n)]
    x = [[mpmath.mpf(float(q[c * n + i])) for c in range(3)] for i in range(n)]
    u = [[mpmath.mpf(float(v[c * n + i])) for c in range(3)] for i in range(n)]
    e2 = mpmath.mpf(EPS) ** 2
    out = {}
    out["mass"] = (sum(me), sum(me))
    kin = sum(me[i] * sum(c * c for c in u[i]) for i in range(n)) / 2
    out["kinetic"] = (kin, kin)
    pot = mpmath.mpf(0)
    for i in range(n):
        for j in range(i + 1, n):
            pot += me[i] * me[j] / mpmath.sqrt(sum((x[j][c] - x[i][c]) ** 2 for c in range(3)) + e2)
    out["potential"] = (-mpmath.mpf(G) * pot, mpmath.mpf(G) * pot)
    for c in range(3):
        t = [me[i] * u[i][c] for i in range(n)]
        out["momentum%d" % c] = (sum(t), sum(abs(a) for a in t))
        a, b = (c + 1) % 3, (c + 2) % 3  # (q x v)_c = q_a v_b - q_b v_a
        t = [me[i] * x[i][a] * u[i][b] for i in range(n)] + [-me[i] * x[i][b] * u[i][a] for i in range(n)]
        out["angular_momentum%d" % c] = (sum(t), sum(abs(s) for s in t))
    return out


def _ld_to_mpf(val):
    import mpmath

    mant, ex = np.frexp(np.longdouble(val))
    return mpmath.mpf(int(np.ldexp(mant, 64))) * mpmath.mpf(2) ** (int(ex) - 64)


def crafted_systems():
    rng = np.random.default_rng(11)
    out = []
    # coincident bodies (r = 0: the term is m m / eps), a pair closer than eps, 1e30 kg beside massless bodies
    x = np.array([[1.0, 2.0, 3.0], [1.0, 2.0, 3.0], [1.0 + 3e-4, 2.0, 3.0], [1e9, -2e9, 5e8], [1e9 + 1e-3, -2e9, 5e8],
                  [-7e12, 3e12, 1e11]])
    vv = rng.normal(0, 1e4, x.shape)
    m = np.array([1e30, 1e30, 0.0, 3e24, 0.0, 1e30])
    out.append(("coincident-heavy-massless", x, vv, m, np.zeros(6, np.uint8), 0))
    # coordinates near 2e20 m (the goldens' scale): q x v cancels in its two products
    n = 9
    x = np.array([-2.0e20, -2.9e20, 1.8e18]) + rng.uniform(-5e12, 5e12, (n, 3))
    vv = rng.normal(0, 1e7, (n, 3))
    m = 10.0 ** rng.uniform(20, 30, n)
    m[3] = 0.0
    out.append(("far-from-origin", x, vv, m, np.zeros(n, np.uint8), 0))
    # gravity devices at a step with |sin| != 0 (and a massless device)
    dev = np.zeros(n, np.uint8)
    dev[[2, 5, 3]] = 1
    out.append(("devices-step-12345", x, vv, m, dev, 12345))
    out.append(("devices-step-1", x * 1e-8, vv, m, dev, 1))
    return out


@pytest.mark.parametrize("label,x,vv,m,dev,step", crafted_systems(), ids=[c[0] for c in crafted_systems()])
def test_reference_diagnostics_against_mpmath(label, x, vv, m, dev, step):
    import mpmath

    n = len(m)
    q = np.ascontiguousarray(x.T).reshape(-1)
    v = np.ascontiguousarray(vv.T).reshape(-1)
    assert fst(step) != 0 or step == 0
    got = diag_reference.diagnostics(n, q, v, m, dev, step)
    want = exact_terms(n, q, v, m, dev, step)
    flat = dict(mass=got["mass"], kinetic=got["kinetic"], potential=got["potential"])
    for c in range(3):
        flat["momentum%d" % c] = got["momentum"][c]
        flat["angular_momentum%d" % c] = got["angular_momentum"][c]
    for k, (val, scale) in want.items():
        err = abs(_ld_to_mpf(flat[k]) - val)
        assert err <= mpmath.mpf(2) ** -60 * scale, (label, k, float(err), float(scale))
    assert float(want["potential"][0]) < 0
    # the reference does not depend on its thread count
    one = diag_reference.diagnostics(n, q, v, m, dev, step, nthreads=1)
    assert all(np.array_equal(np.atleast_1d(one[k]), np.atleast_1d(got[k])) for k in got)


def test_nb_diag_layout_matches_header(nb, tmp_path):
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "nbody_b200.h"\n'
                   'int main(){printf("%zu %zu %zu %zu %zu %zu %zu\\n", sizeof(nb_diag), offsetof(nb_diag, n), '
                   'offsetof(nb_diag, mass), offsetof(nb_diag, kinetic), offsetof(nb_diag, potential), '
                   'offsetof(nb_diag, momentum), offsetof(nb_diag, angular_momentum));return 0;}\n')
    exe = tmp_path / "layout"
    subprocess.check_call(["/usr/bin/gcc", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)])
    got = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    D = nb.NbDiag
    assert got == [C.sizeof(D), D.n.offset, D.mass.offset, D.kinetic.offset, D.potential.offset, D.momentum.offset,
                   D.angular_momentum.offset]
    assert got[0] == 80


def test_diagnostics_argument_validation(nb):
    L = nb.lib()
    q, m = np.zeros(3), np.zeros(1)
    dev = np.zeros(1, np.uint8)
    out = nb.NbDiag()
    ok = (nb._d(q), nb._d(q), nb._d(m), nb._u(dev))
    call = lambda S, n, arrays, step, o: L.nb_diagnostics(0, S, n, *arrays, step, o, None)
    assert call(1, 0, ok, 0, C.byref(out)) == nb.NB_ERR_ARG          # n < 1
    assert call(0, 1, ok, 0, C.byref(out)) == nb.NB_ERR_ARG          # n_systems < 1
    assert call(1, 1, ok, -1, C.byref(out)) == nb.NB_ERR_ARG         # step < 0
    assert call(1, 1, ok, 0, None) == nb.NB_ERR_ARG                  # null output
    for k in range(4):                                              # each null input
        arrays = list(ok)
        arrays[k] = None
        assert call(1, 1, arrays, 0, C.byref(out)) == nb.NB_ERR_ARG
    assert L.nb_traj_diagnostics(None, C.byref(out)) == nb.NB_ERR_ARG
    with pytest.raises(ValueError):
        nb.diagnostics(np.zeros(4), np.zeros(4), np.zeros(1), np.zeros(1, np.uint8))


def test_diagnostics_without_gpu_fails_loudly(nb):
    if nb.device_count() > 0:
        pytest.skip("a GPU is present")
    s = nb.generate_system(16, seed=1)
    with pytest.raises(nb.NbodyError) as e:
        nb.diagnostics(s.q, s.v, s.m, s.is_device)
    assert e.value.code == nb.NB_ERR_NO_GPU
    with pytest.raises(nb.NbodyError) as e:
        nb.diagnostics(np.stack([s.q, s.q]), np.stack([s.v, s.v]), np.stack([s.m, s.m]),
                       np.stack([s.is_device, s.is_device]), step=5)
    assert e.value.code == nb.NB_ERR_NO_GPU


def test_nbtool_diag_without_file_prints_usage(nb):
    r = subprocess.run([nb.NBTOOL_PATH, "diag"], capture_output=True, text=True)
    assert r.returncode == 2 and "nbtool diag <in> [step]" in r.stderr


LIB = os.path.join(ROOT, "nthu_ipc_nbody-simulation_b200", "libnbody_b200.so")


@pytest.mark.skipif(shutil.which("cuobjdump") is None or not os.path.exists(LIB), reason="cuobjdump or the library is missing")
def test_diag_kernels_in_library():
    out = subprocess.check_output(["cuobjdump", "-sass", LIB]).decode()
    funcs = {}
    for b in re.split(r"\n\s*Function : ", out)[1:]:
        name, body = b.split("\n", 1)
        funcs[name.strip()] = body
    pot = [b for k, b in funcs.items() if "sym_potential_kernel" in k]
    red = [b for k, b in funcs.items() if "sym_diag_sum_kernel" in k]
    assert len(pot) == 1 and len(red) == 1
    assert "MUFU.RSQ64H" in pot[0] and re.search(r"\bDFMA\b", pot[0])
    for body in pot + red:
        assert "ATOM" not in body and "RED." not in body


def test_diag_kernels_do_not_spill():
    log = os.path.join(ROOT, "nthu_ipc_nbody-simulation_b200", "_build", "nb_diag.ptxas.log")
    if not os.path.exists(log):
        pytest.skip("ptxas log not kept")
    text = open(log).read()
    props = re.findall(r"Function properties for (\S+)\n\s*(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads",
                       text)
    names = [p[0] for p in props]
    assert any("sym_potential_kernel" in x for x in names) and any("sym_diag_sum_kernel" in x for x in names)
    for name, _, st, ld in props:
        assert st == "0" and ld == "0", name
