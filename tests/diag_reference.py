"""ctypes binding of tests/diag_reference.cc, the long-double reference of the diagnostics (test infrastructure only).

The shared library is compiled on first use into a temporary directory, never into the tree."""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "diag_reference.cc")
_lib = None


def _compiler():
    return "/usr/bin/g++" if os.access("/usr/bin/g++", os.X_OK) else "g++"


def lib():
    global _lib
    if _lib is None:
        d = tempfile.mkdtemp(prefix="diag_reference_")
        atexit.register(shutil.rmtree, d, True)
        so = os.path.join(d, "libdiag_reference.so")
        base = [_compiler(), "-O2", "-std=c++17", "-ffp-contract=off", "-shared", "-fPIC", "-o", so, SRC]
        # OpenMP over the rows when the toolchain has it (the result does not depend on it)
        if subprocess.run(base[:1] + ["-fopenmp"] + base[1:], capture_output=True).returncode != 0:
            subprocess.check_call(base)
        L = C.CDLL(so)
        L.diag_reference.argtypes = [C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_double),
                                     C.POINTER(C.c_ubyte), C.c_int, C.c_int, C.POINTER(C.c_longdouble)]
        _lib = L
    return _lib


def _d(a):
    a = np.ascontiguousarray(a, dtype=np.float64)
    return a, a.ctypes.data_as(C.POINTER(C.c_double))


def diagnostics(n, q, v, m, is_device, step=0, nthreads=None):
    """The quantities of nb_diag in long double (compensated sums), as a dict of np.longdouble
    (momentum, angular_momentum: arrays of 3)."""
    assert np.finfo(np.longdouble).nmant >= 63, "the reference needs an extended long double"
    assert C.sizeof(C.c_longdouble) == np.dtype(np.longdouble).itemsize
    nthreads = nthreads or os.cpu_count()
    q, qp = _d(q)
    v, vp = _d(v)
    m, mp = _d(m)
    dev = np.ascontiguousarray(is_device, dtype=np.uint8)
    r = np.zeros(9, dtype=np.longdouble)
    rc = lib().diag_reference(n, qp, vp, mp, dev.ctypes.data_as(C.POINTER(C.c_ubyte)), step, nthreads,
                              r.ctypes.data_as(C.POINTER(C.c_longdouble)))
    assert rc == 0
    return dict(mass=r[0], kinetic=r[1], potential=r[2], momentum=r[3:6].copy(), angular_momentum=r[6:9].copy())
