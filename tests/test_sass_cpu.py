"""Build evidence that needs no GPU: the built library is sm_100a only and its kernels contain the instructions the design
rests on (1-D TMA bulk copies, cluster multicast, 256-bit sector accesses, register re-allocation between warp roles), read
with cuobjdump.  Skipped when the CUDA binary utilities are not installed."""
import importlib
import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "nthu_ipc_nbody-simulation_b200", "libnbody_b200.so")

pytestmark = pytest.mark.skipif(shutil.which("cuobjdump") is None or not os.path.exists(LIB),
                                reason="cuobjdump or the built library is missing")


@pytest.fixture(scope="module")
def sass():
    out = subprocess.check_output(["cuobjdump", "-sass", LIB]).decode()
    funcs = {}
    for b in re.split(r"\n\s*Function : ", out)[1:]:
        name, body = b.split("\n", 1)
        funcs[name.strip()] = body
    return out, funcs


def test_only_sm_100a_cubins(sass):
    out, _ = sass
    archs = set(re.findall(r"arch = (sm_\w+)", out))
    assert archs == {"sm_100a"}, archs


def test_grid_kernel_instructions(sass):
    _, funcs = sass
    grid = {k: v for k, v in funcs.items() if "grid_traj_kernel" in k}
    assert len(grid) == 4  # one and two systems per launch, each with and without the phase profile
    for name, body in grid.items():
        assert "UBLKCP" in body and "MULTICAST" in body, name      # TMA bulk copy, multicast into the cluster
        assert "ENL2.256" in body, name                             # one 32-byte sector per record access
        assert "UCGABAR" in body, name                              # cluster barrier around the multicast lifetime
        assert "MUFU.RSQ64H" in body and "DFMA" in body, name
        assert body.count("USETMAXREG") == 2, name                  # registers re-allocated between compute and helper warps
    # two systems in lock step: the compute warps arrive at the integrator warp's barrier
    two = [v for k, v in grid.items() if "grid_traj_kernelILi2E" in k]
    assert len(two) == 2 and all("BAR.ARV" in b for b in two)


def test_no_tensor_core_or_library_kernels(sass):
    """The pair term is not a contraction (north star): no tensor-core instruction anywhere, and every kernel in the library is
    one of this repository's."""
    out, funcs = sass
    assert not re.search(r"\b(HMMA|IMMA|DMMA|UTCHMMA|UTCQMMA|UTMALDG)\b", out)
    own = ("traj_kernel", "traj_sym_kernel", "grid_traj_kernel", "large_", "sym_", "counter_wait_kernel", "dfma_")
    assert all(any(o in name for o in own) for name in funcs), [n for n in funcs if not any(o in n for o in own)]


def test_symmetric_kernels_use_tma_and_no_atomics_on_the_accumulation(sass):
    _, funcs = sass
    for name, body in funcs.items():
        if "sym_accel_kernel" in name:
            assert "UBLKCP" in body and "SHFL.IDX" in body, name
            assert "ATOM" not in body.replace("ATOMS.CAST", ""), name   # partial rows + fixed-order sums, never atomics
            assert len(re.findall(r"\bDFMA\b", body)) >= 400, name


def test_large_n_kernels_are_built_in_the_kept_variants_only(sass):
    """The row kernel exists once per math mode (FAST, STRICT; 4 i-bodies per thread is a constant), the symmetric kernel
    once per row width (6 and 8 i-bodies per lane, chosen by shard size).  No other variant is built."""
    _, funcs = sass
    targs = lambda kernel: sorted(re.search(kernel + r"I(\w+?)EEv", k).group(1) for k in funcs if kernel in k)
    assert targs("large_accel_kernel") == ["Li0E", "Li1E"], targs("large_accel_kernel")  # <MATH_FAST>, <MATH_STRICT>
    assert targs("sym_accel_kernel") == ["Li6E", "Li8E"], targs("sym_accel_kernel")


def test_grid_pair_loop_schedule_did_not_regress():
    """The pair loop of the grid kernel is the one place where ptxas' register allocation decides the speed: with the role
    branches not dominated by their setmaxnreg it once scheduled 668 stall cycles per 8 pairs instead of 320 (4.2 us per step
    instead of 3.3).  Guard: the production instantiations (one system; two systems in lock step) stay below 340."""
    import sys
    obj = os.path.join(ROOT, "nthu_ipc_nbody-simulation_b200", "_build", "nb_grid.o")
    if not os.path.exists(obj):
        pytest.skip("object file not kept")
    for inst in ("grid_traj_kernelILi1ELb0E", "grid_traj_kernelILi2ELb0E"):
        out = subprocess.check_output([sys.executable, os.path.join(ROOT, "tools", "sass_loop_stalls.py"), obj, inst, "120"]).decode()
        loops = [(int(m.group(1)), int(m.group(2))) for m in re.finditer(r"(\d+) FP64, sum of stall counts (\d+)", out)]
        pair_loops = [s for n, s in loops if n == 128]  # 8 pairs x 16 FP64 instructions per trip
        assert pair_loops, out
        assert max(pair_loops) <= 340, (inst, pair_loops)
