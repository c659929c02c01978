"""nbody_b200 — B200 (sm_100a) implementation of the N-body hot path of
dasbd72/NTHU_IPC_Nbody-Simulation, behind the C ABI declared in include/nbody_b200.h.

This Python layer is a thin ctypes mirror of that ABI (used by the tests, bench.py and the
sharded multi-GPU driver).  The product is libnbody_b200.so + the `hw5` CLI; there is NO CPU
fallback: importing works anywhere, computing without the built library or without a GPU raises.

Names follow the reference: run_step (samples/nbody.cc:51), read_input / write_output
(nbody.cc:22-49), the three problems of main() (nbody.cc:106-143, hw5.cu:532-616).
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("NB_LIB_PATH") or os.path.join(_HERE, "libnbody_b200.so")  # NB_LIB_PATH: A/B builds of the library
NBTOOL_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "nbtool")
HW5_PATH = os.path.join(_HERE, "hw5")

NB_OK = 0
NB_ERR_ARG, NB_ERR_CUDA, NB_ERR_NO_GPU, NB_ERR_UNSUPPORTED, NB_ERR_IO = -1, -2, -3, -4, -5
MATH_FAST, MATH_STRICT = 0, 1
SOLVE_ALL_DEVICES = 0x100  # OR into math: every device's query-3 trajectory from step 0 (NB_SOLVE_ALL_DEVICES)
KIND_PLAIN, KIND_Q1, KIND_Q2, KIND_Q3 = 0, 1, 2, 3
MAX_DEVICES = 64
MAX_SMALL_N = 1024
N_STEPS = 200000
DT = 60.0
PAIR_FLOPS = 20  # algorithmic flops per ordered pair interaction (SURVEY.md §8d)


class NbodyError(RuntimeError):
    def __init__(self, code, detail=""):
        self.code = code
        super().__init__("nbody_b200 error %d: %s%s" % (code, _strerror(code), (" — " + detail) if detail else ""))


class NbSystem(C.Structure):
    _fields_ = [("n", C.c_int), ("planet", C.c_int), ("asteroid", C.c_int), ("q", C.POINTER(C.c_double)),
                ("v", C.POINTER(C.c_double)), ("m", C.POINTER(C.c_double)), ("is_device", C.POINTER(C.c_ubyte))]


class NbEvents(C.Structure):
    _fields_ = [("min_d2", C.c_double), ("argmin_step", C.c_int), ("hit_step", C.c_int),
                ("destroyed_step", C.c_int), ("cost", C.c_double), ("steps_done", C.c_int), ("n_reach", C.c_int),
                ("reach_step", C.c_int * MAX_DEVICES)]

    def as_dict(self):
        return dict(min_d2=self.min_d2, argmin_step=self.argmin_step, hit_step=self.hit_step,
                    destroyed_step=self.destroyed_step, cost=self.cost, steps_done=self.steps_done,
                    reach_step=list(self.reach_step[: self.n_reach]))


class NbAnswer(C.Structure):
    _fields_ = [("min_dist", C.c_double), ("hit_time_step", C.c_int), ("gravity_device_id", C.c_int),
                ("missile_cost", C.c_double), ("argmin_step", C.c_int), ("n_devices", C.c_int),
                ("device_index", C.c_int * MAX_DEVICES), ("reach_step", C.c_int * MAX_DEVICES),
                ("q3_hit_step", C.c_int * MAX_DEVICES), ("q3_cost", C.c_double * MAX_DEVICES),
                ("gpu_seconds", C.c_double), ("wall_seconds", C.c_double), ("pair_interactions", C.c_longlong),
                ("n_trajectories", C.c_int), ("n_gpus_used", C.c_int)]


# every symbol include/nbody_b200.h declares (tests/test_abi.py checks the two lists agree)
ABI_SYMBOLS = [
    "nb_version", "nb_strerror", "nb_last_error_detail", "nb_device_count", "nb_kernel_launches", "nb_grid_torn_records",
    "nb_run_steps", "nb_traj_create", "nb_traj_run", "nb_traj_state", "nb_traj_fork", "nb_traj_fork_on", "nb_traj_destroy",
    "nb_ensemble_run", "nb_solve", "nb_solve_trajectory_count", "nb_solve_partial", "nb_solve_combine",
    "nb_profile_enable", "nb_profile_read", "nb_read_header", "nb_read_input", "nb_write_output", "nb_write_input", "nb_generate_system", "nb_hw5_main",
    "nb_large_scratch_bytes", "nb_large_pack", "nb_large_unpack", "nb_large_step", "nb_large_step_p2p", "nb_large_blocks_per_step", "nb_large_p2p_counter_bytes", "nb_large_wait_p2p",
    "nb_dev_alloc", "nb_dev_free", "nb_dev_copy", "nb_ipc_export", "nb_ipc_open", "nb_ipc_close", "nb_fp64_peak", "nb_fp64_peak_variant",
    "nb_sym_create", "nb_sym_destroy", "nb_sym_pj_bytes", "nb_sym_counter_bytes", "nb_sym_blocks", "nb_sym_remote_partial_bytes",
    "nb_sym_pairs", "nb_sym_wait_positions", "nb_sym_step", "nb_sym_step_phase", "nb_sym_plan_describe", "nb_sym_rows", "nb_sym_row_size", "nb_sym_row_stride", "nb_device_warm", "nb_hw5_narrow_visible_gpus", "nb_sym_publish_rows", "nb_sym_unpack_rows", "nb_sym_step_host",
]


_lib_handle = None
_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)
_up = C.POINTER(C.c_ubyte)


def lib():
    """The loaded C-ABI library.  Fails loudly when it has not been built (no fallback)."""
    global _lib_handle
    if _lib_handle is not None:
        return _lib_handle
    if not os.path.exists(LIB_PATH):
        raise ImportError("libnbody_b200.so is not built: run `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(or make -C %s/csrc); there is no CPU fallback" % _HERE)
    L = C.CDLL(LIB_PATH)
    L.nb_version.restype = C.c_char_p
    L.nb_strerror.restype = C.c_char_p
    L.nb_strerror.argtypes = [C.c_int]
    L.nb_last_error_detail.restype = C.c_char_p
    L.nb_device_count.argtypes = [_ip]
    L.nb_kernel_launches.restype = C.c_longlong
    L.nb_grid_torn_records.restype = C.c_longlong
    L.nb_run_steps.argtypes = [C.c_int, C.c_int, C.c_int, _dp, _dp, _dp, _up, C.c_int, C.c_int]
    L.nb_traj_create.argtypes = [C.c_int, C.POINTER(NbSystem), C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p)]
    L.nb_traj_run.argtypes = [C.c_void_p, C.c_int, C.POINTER(NbEvents)]
    L.nb_traj_state.argtypes = [C.c_void_p, _dp, _dp, _dp, _ip]
    L.nb_traj_fork.argtypes = [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_void_p)]
    L.nb_traj_fork_on.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p)]
    L.nb_traj_destroy.argtypes = [C.c_void_p]
    L.nb_ensemble_run.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _dp, _dp, _dp, _up, _ip, _ip, _ip,
                                  C.c_int, C.c_int, C.POINTER(NbEvents), _dp]
    L.nb_solve.argtypes = [C.POINTER(NbSystem), _ip, C.c_int, C.c_int, C.c_int, C.POINTER(NbAnswer)]
    L.nb_solve_trajectory_count.argtypes = [C.POINTER(NbSystem), _ip]
    L.nb_solve_partial.argtypes = [C.POINTER(NbSystem), C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                   C.POINTER(NbEvents), _dp, C.POINTER(C.c_longlong)]
    L.nb_solve_combine.argtypes = [C.POINTER(NbSystem), C.POINTER(NbEvents), C.POINTER(NbAnswer)]
    L.nb_profile_enable.argtypes = [C.c_int]
    L.nb_profile_read.argtypes = [_dp, C.POINTER(C.c_longlong)]
    L.nb_read_header.argtypes = [C.c_char_p, _ip, _ip, _ip]
    L.nb_read_input.argtypes = [C.c_char_p, C.c_int, _ip, _ip, _ip, _dp, _dp, _dp, _up]
    L.nb_write_output.argtypes = [C.c_char_p, C.c_double, C.c_int, C.c_int, C.c_double]
    L.nb_hw5_main.argtypes = [C.c_char_p, C.c_char_p, C.c_int]
    L.nb_write_input.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_int, _dp, _dp, _dp, _up]
    L.nb_generate_system.argtypes = [C.c_int, C.c_ulonglong, C.c_int, _dp, _dp, _dp, _up, _ip, _ip]
    L.nb_large_scratch_bytes.restype = C.c_longlong
    L.nb_large_scratch_bytes.argtypes = [C.c_int, C.c_int]
    L.nb_large_pack.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    L.nb_large_unpack.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    L.nb_large_step.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.nb_large_step_p2p.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.POINTER(C.c_void_p),
                                    C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_ulonglong, C.c_void_p, C.c_void_p,
                                    C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.nb_large_blocks_per_step.argtypes = [C.c_int]
    L.nb_large_wait_p2p.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_ulonglong, C.c_void_p, C.c_void_p]
    L.nb_dev_alloc.argtypes = [C.c_longlong, C.POINTER(C.c_void_p)]
    L.nb_dev_free.argtypes = [C.c_void_p]
    L.nb_dev_copy.argtypes = [C.c_void_p, C.c_void_p, C.c_longlong, C.c_int, C.c_void_p]
    L.nb_ipc_export.argtypes = [C.c_void_p, C.c_char_p]
    L.nb_ipc_open.argtypes = [C.c_char_p, C.POINTER(C.c_void_p)]
    L.nb_ipc_close.argtypes = [C.c_void_p]
    L.nb_sym_create.argtypes = [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p)]
    L.nb_sym_destroy.argtypes = [C.c_void_p]
    L.nb_sym_pj_bytes.restype = C.c_longlong
    L.nb_sym_pj_bytes.argtypes = [C.c_void_p]
    L.nb_sym_blocks.argtypes = [C.c_void_p]
    L.nb_sym_remote_partial_bytes.restype = C.c_longlong
    L.nb_sym_remote_partial_bytes.argtypes = [C.c_void_p]
    L.nb_sym_pairs.restype = C.c_longlong
    L.nb_sym_pairs.argtypes = [C.c_void_p, C.POINTER(C.c_longlong), C.POINTER(C.c_longlong)]
    L.nb_sym_wait_positions.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.nb_sym_step.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p),
                              C.POINTER(C.c_void_p), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.nb_sym_step_phase.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p),
                                    C.POINTER(C.c_void_p), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.nb_sym_publish_rows.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p),
                                      C.c_void_p, C.c_void_p, C.c_void_p]
    L.nb_sym_unpack_rows.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.nb_sym_step_host.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p),
                                   C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_void_p, C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.c_void_p]
    L.nb_sym_plan_describe.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _ip, _ip, _ip, _ip, _ip, C.c_int,
                                       C.POINTER(C.c_longlong), C.POINTER(C.c_longlong)]
    L.nb_sym_rows.argtypes = [C.c_int, C.c_int]
    L.nb_sym_row_stride.argtypes = [C.c_int, C.c_int]
    L.nb_fp64_peak.argtypes = [C.c_int, _dp, _dp]
    L.nb_fp64_peak_variant.argtypes = [C.c_int, C.c_int, _dp]
    _lib_handle = L
    return L


def _strerror(code):
    try:
        return lib().nb_strerror(code).decode()
    except Exception:
        return "?"


def _check(rc):
    if rc != NB_OK:
        raise NbodyError(rc, lib().nb_last_error_detail().decode())


def _d(a):
    return a.ctypes.data_as(_dp)


def _u(a):
    return a.ctypes.data_as(_up)


def _i(a):
    return a.ctypes.data_as(_ip)


@dataclass
class System:
    """One input file: planar q[3n], v[3n] (x block, y block, z block), m[n], is_device[n]."""
    n: int
    planet: int
    asteroid: int
    q: np.ndarray
    v: np.ndarray
    m: np.ndarray
    is_device: np.ndarray

    def copy(self):
        return System(self.n, self.planet, self.asteroid, self.q.copy(), self.v.copy(), self.m.copy(),
                      self.is_device.copy())

    @property
    def devices(self):
        return [int(i) for i in np.nonzero(self.is_device)[0]]

    def _c(self):
        for a in (self.q, self.v, self.m):
            assert a.dtype == np.float64 and a.flags.c_contiguous
        assert self.is_device.dtype == np.uint8
        return NbSystem(self.n, self.planet, self.asteroid, _d(self.q), _d(self.v), _d(self.m), _u(self.is_device))


def device_count():
    c = C.c_int(0)
    rc = lib().nb_device_count(C.byref(c))
    return c.value if rc == NB_OK else 0


def kernel_launches():
    return int(lib().nb_kernel_launches())


def grid_torn_records():
    """Torn 32-byte records the grid kernel's exchange detected and fetched again in this process (expected 0)."""
    return int(lib().nb_grid_torn_records())


def read_input(path):
    """nbody.cc:22-39 / hw5.cu:86-131 (without the reference's body permutation)."""
    n, p, a = C.c_int(), C.c_int(), C.c_int()
    _check(lib().nb_read_header(os.fsencode(path), C.byref(n), C.byref(p), C.byref(a)))
    nn = n.value
    q, v, m = np.empty(3 * nn), np.empty(3 * nn), np.empty(nn)
    dev = np.zeros(nn, dtype=np.uint8)
    _check(lib().nb_read_input(os.fsencode(path), nn, C.byref(n), C.byref(p), C.byref(a), _d(q), _d(v), _d(m), _u(dev)))
    return System(nn, p.value, a.value, q, v, m, dev)


def write_input(path, s):
    """The reference's input format (nbody.cc:22-39), written with 17 significant digits."""
    _check(lib().nb_write_input(os.fsencode(path), s.n, s.planet, s.asteroid, _d(s.q), _d(s.v), _d(s.m), _u(s.is_device)))


def generate_system(n, seed=42, n_devices=4):
    """SURVEY.md 8d config C5 (std::mt19937_64(seed) in the library, same as `nbtool gen n seed out.in`): positions
    uniform in a cube of side 1e13 m centred at (-2.0e20, -2.9e20, 1.8e18), velocities N(0, (1e7 m/s)^2), masses
    log-uniform in [1e20, 1e30] kg, body 0 = planet, body 1 = asteroid, the last n_devices bodies gravity devices."""
    q, v, m = np.empty(3 * n), np.empty(3 * n), np.empty(n)
    dev = np.zeros(n, dtype=np.uint8)
    p, a = C.c_int(), C.c_int()
    _check(lib().nb_generate_system(n, seed, n_devices, _d(q), _d(v), _d(m), _u(dev), C.byref(p), C.byref(a)))
    return System(n, p.value, a.value, q, v, m, dev)


def write_output(path, min_dist, hit_time_step, gravity_device_id, missile_cost):
    """nbody.cc:41-49."""
    _check(lib().nb_write_output(os.fsencode(path), min_dist, hit_time_step, gravity_device_id, missile_cost))


def run_step(step, n, q, v, m, is_device, gpu=0, math=MATH_FAST):
    """run_step(step, n, q.., v.., m, type) of nbody.cc:51-89 on planar host arrays, in place."""
    run_steps(step - 1, step, n, q, v, m, is_device, gpu=gpu, math=math)


def run_steps(step_begin, step_end, n, q, v, m, is_device, gpu=0, math=MATH_FAST):
    """Steps step_begin+1 .. step_end on planar HOST arrays, in place (H2D, kernels, D2H)."""
    _check(lib().nb_run_steps(gpu, math, n, _d(q), _d(v), _d(m), _u(is_device), step_begin, step_end))


class Trajectory:
    """One persistent-kernel trajectory (hw5.cu:322-436 / 438-530 inner loops)."""

    def __init__(self, system, kind, destroy_device=-1, gpu=0, math=MATH_FAST, _handle=None):
        self._h = C.c_void_p()
        self.n = system.n if system is not None else None
        if _handle is not None:
            self._h = _handle
            return
        cs = system._c()
        _check(lib().nb_traj_create(gpu, C.byref(cs), kind, destroy_device, math, C.byref(self._h)))

    def run(self, step_end):
        ev = NbEvents()
        _check(lib().nb_traj_run(self._h, step_end, C.byref(ev)))
        return ev

    def state(self):
        q, v, m = np.empty(3 * self.n), np.empty(3 * self.n), np.empty(self.n)
        step = C.c_int()
        _check(lib().nb_traj_state(self._h, _d(q), _d(v), _d(m), C.byref(step)))
        return q, v, m, step.value

    def fork(self, kind, destroy_device=-1, gpu=None):
        h = C.c_void_p()
        if gpu is None:
            _check(lib().nb_traj_fork(self._h, kind, destroy_device, C.byref(h)))
        else:
            _check(lib().nb_traj_fork_on(self._h, gpu, kind, destroy_device, C.byref(h)))
        t = Trajectory(None, kind, _handle=h)
        t.n = self.n
        return t

    def close(self):
        if self._h:
            lib().nb_traj_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def ensemble_run(q, v, m, is_device, planet, asteroid, kind=KIND_PLAIN, destroy_device=None, step_begin=0,
                 step_end=1, gpu=0, math=MATH_FAST):
    """S systems of the same n in one launch.  q, v: [S, 3n] (updated in place); m: [S, n];
    is_device: [S, n] uint8; planet / asteroid / destroy_device: [S] int32.  Returns (events, gpu_seconds)."""
    S, n3 = q.shape
    n = n3 // 3
    ev = (NbEvents * S)()
    secs = C.c_double(0)
    planet = np.ascontiguousarray(planet, dtype=np.int32)
    asteroid = np.ascontiguousarray(asteroid, dtype=np.int32)
    dd = None if destroy_device is None else np.ascontiguousarray(destroy_device, dtype=np.int32)
    _check(lib().nb_ensemble_run(gpu, math, kind, S, n, _d(q), _d(v), _d(m), _u(is_device), _i(planet), _i(asteroid),
                                 _i(dd) if dd is not None else None, step_begin, step_end, ev, C.byref(secs)))
    return list(ev), secs.value


def solve(system, gpus=None, n_steps=N_STEPS, math=MATH_FAST, all_devices=False):
    """The three problems of main() (nbody.cc:106-143, hw5.cu:563-606) -> NbAnswer.  With fewer GPUs than trajectories
    the scheduler forks query 3 from query 2 and stops at the cheapest saving device (q3_hit_step == -3 for devices it
    did not need to simulate); all_devices=True simulates every device's trajectory from step 0."""
    if all_devices:
        math |= SOLVE_ALL_DEVICES
    if gpus is None:
        gpus = [0]
    if isinstance(gpus, int):
        gpus = list(range(gpus))
    g = np.ascontiguousarray(gpus, dtype=np.int32)
    ans = NbAnswer()
    cs = system._c()
    _check(lib().nb_solve(C.byref(cs), _i(g), len(g), n_steps, math, C.byref(ans)))
    return ans


def solve_partial(system, gpu, part, n_parts, n_steps=N_STEPS, math=MATH_FAST, all_devices=False):
    """This part's share of the trajectories on `gpu` (the library's scheduler decides which: nb_host.cu).
    Returns (events array: this part's entries filled, the others marked steps_done == -2; gpu_seconds; pair_interactions)."""
    if all_devices:
        math |= SOLVE_ALL_DEVICES
    cs = system._c()
    cnt = C.c_int()
    _check(lib().nb_solve_trajectory_count(C.byref(cs), C.byref(cnt)))
    evs = (NbEvents * cnt.value)()
    secs, pairs = C.c_double(), C.c_longlong()
    _check(lib().nb_solve_partial(C.byref(cs), gpu, part, n_parts, n_steps, math, evs, C.byref(secs), C.byref(pairs)))
    return evs, secs.value, pairs.value


def solve_combine(system, evs):
    cs = system._c()
    ans = NbAnswer()
    _check(lib().nb_solve_combine(C.byref(cs), evs, C.byref(ans)))
    return ans


def solve_distributed(system, rank, world, gpu, n_steps=N_STEPS, math=MATH_FAST, group=None, all_devices=False):
    """One process per GPU (torchrun): every rank simulates its share of the trajectories, the
    nb_events structs (a few hundred bytes each) are gathered with torch.distributed — the path has
    no data-path collective — and every rank applies the selection rule.  Returns (answer,
    max gpu_seconds over ranks, total pair interactions)."""
    evs, secs, pairs = solve_partial(system, gpu, rank, world, n_steps, math, all_devices)
    if world > 1:
        import torch.distributed as dist

        blobs = [None] * world
        dist.all_gather_object(blobs, (bytes(evs), secs, pairs), group=group)
        T = len(evs)
        merged = (NbEvents * T)()
        for r, (b, s_r, p_r) in enumerate(blobs):
            part = (NbEvents * T).from_buffer_copy(b)
            for t in range(T):
                if part[t].steps_done != -2:  # -2 = another part's trajectory
                    merged[t] = part[t]
        evs = merged
        secs = max(b[1] for b in blobs)
        pairs = sum(b[2] for b in blobs)
    return solve_combine(system, evs), secs, pairs


def sym_plan(n, world, rank, blocks):
    """The static schedule of the symmetric large-N stepper for one rank (host only, csrc/nb_sym.cu build_plan):
    returns (segs[k, 8] = {row_body0, row_count, j0, j1, flags, pi_slot, pj_row, src_rank}, block_seg_begin[blocks+1],
    pj_ptr[rows+1], pj_list, symmetric unordered pairs, one-sided ordered pairs)."""
    L = lib()
    ns, sp, op = C.c_int(), C.c_longlong(), C.c_longlong()
    _check(L.nb_sym_plan_describe(n, world, rank, blocks, 0, None, C.byref(ns), None, None, None, 0, C.byref(sp), C.byref(op)))
    segs = np.zeros((max(ns.value, 1), 8), dtype=np.int32)
    bsb = np.zeros(blocks + 1, dtype=np.int32)
    rows = L.nb_sym_rows(n, world)
    pj_ptr = np.zeros(rows + 1, dtype=np.int32)
    max_pj = rows * rows * world + 1
    pj_list = np.zeros(max_pj, dtype=np.int32)
    _check(L.nb_sym_plan_describe(n, world, rank, blocks, len(segs), _i(segs), C.byref(ns), _i(bsb), _i(pj_ptr), _i(pj_list),
                                  max_pj, C.byref(sp), C.byref(op)))
    return segs[: ns.value], bsb, pj_ptr, pj_list[: pj_ptr[-1]], sp.value, op.value


def profile_enable(on=True):
    _check(lib().nb_profile_enable(1 if on else 0))


def profile_read():
    ms, cnt = C.c_double(), C.c_longlong()
    _check(lib().nb_profile_read(C.byref(ms), C.byref(cnt)))
    return ms.value, cnt.value


def format_output(min_dist, hit_time_step, gravity_device_id, missile_cost):
    return "%.16e\n%d\n%d %.16e\n" % (min_dist, hit_time_step, gravity_device_id, missile_cost)


def hw5_main(input_path, output_path, n_gpus=0):
    """hw5 <input> <output> through the library entry point (the `hw5` binary calls the same)."""
    _check(lib().nb_hw5_main(os.fsencode(input_path), os.fsencode(output_path), n_gpus))


def fp64_peak(gpu=0, variant=0):
    t, s = C.c_double(), C.c_double()
    if variant:
        _check(lib().nb_fp64_peak_variant(gpu, variant, C.byref(t)))
    else:
        _check(lib().nb_fp64_peak(gpu, C.byref(t), C.byref(s)))
    return t.value


from .sharded import P2PShardedSystem, ShardedSystem, SymLocalWorld, SymShardedSystem, partition, synthetic_system  # noqa: E402,F401
