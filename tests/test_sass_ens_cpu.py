"""Build evidence without a GPU for the ensemble kernels of n > 1024 bodies (nb_ens.cu), read with cuobjdump: each kernel is
built once, the FAST tile kernel is the shuffle-rotation pair loop on the rsqrt seed, and no kernel sums with atomics."""
import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "nthu_ipc_nbody-simulation_b200", "libnbody_b200.so")
KERNELS = ("sym_ens_tile_kernel", "large_ens_strict_kernel", "large_ens_integrate_kernel", "large_ens_observe_kernel")

pytestmark = pytest.mark.skipif(shutil.which("cuobjdump") is None or not os.path.exists(LIB),
                                reason="cuobjdump or the built library is missing")


@pytest.fixture(scope="module")
def funcs():
    out = subprocess.check_output(["cuobjdump", "-sass", LIB]).decode()
    f = {}
    for b in re.split(r"\n\s*Function : ", out)[1:]:
        name, body = b.split("\n", 1)
        f[name.strip()] = body
    return f


def test_each_ensemble_kernel_is_built_once(funcs):
    for k in KERNELS:
        assert sum(k in name for name in funcs) == 1, (k, [n for n in funcs if k in n])


def test_tile_kernel_is_the_symmetric_rsqrt_pair_loop(funcs):
    (body,) = [b for n, b in funcs.items() if "sym_ens_tile_kernel" in n]
    assert "SHFL" in body and "MUFU.RSQ64H" in body and re.search(r"\bDFMA\b", body)


def test_no_atomics_in_the_ensemble_kernels(funcs):
    for name, body in funcs.items():
        if any(k in name for k in KERNELS):
            assert not re.search(r"\b(ATOM|ATOMG|ATOMS|RED|REDG|REDUX)\b", body), name
