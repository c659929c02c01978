#!/usr/bin/env python
"""bench.py — the driver's measurement contract for the N-body hot path.

    python bench.py --gpus N --steps K --warmup W            (N>1: launched under torchrun, one rank per GPU)
    python bench.py --impl reference --steps K --warmup W    (the reference's own CPU program)

Metric (BASELINE.json): FP64 pair-interactions per second on the synthetic 65 536-body single system
(SURVEY.md §8d config C5), body-sharded over the N ranks with a per-step in-place NCCL all-gather of
the 32-byte pos4 records (strong scaling: the total work is fixed).  One "step" = one time step of
the whole system = n(n-1) ordered pair interactions.  The b1024 three-query end-to-end seconds —
the other half of the BASELINE metric — is reported in the same line under "b1024".

    value     pairs/s, device-resident state, CUDA events per step, max over ranks
    e2e       the same metric through the run_step operator with HOST (pinned) buffers: every step
              copies q (all bodies) and this rank's v host->device and back
    roofline  the acceleration kernel alone against the B200 FP64 peak (20 flop per pair)
    cpu_baseline  the unmodified reference program (oracle/_ref/nbody = samples/nbody.cc) on one host
              core, full b20 run (N=1, rank 0 only)

--dump-outputs DIR writes the state the timed steps left (positions.npy, velocities.npy) so that two builds run
with the same arguments can be compared output for output: the input system is generated from a fixed seed.
"""
import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
PKG = "nthu_ipc_nbody-simulation_b200"
CASES = os.path.join(ROOT, "tests", "golden", "testcases")
FP64_PEAK_NOMINAL_TFLOPS = 148 * 64 * 2 * 1.965e9 / 1e12  # 37.2: 148 SM x 64 FMA/clk x 2 x 1.965 GHz
PAIR_FLOPS = 20
METRIC = "fp64_pair_interactions_per_sec"
UNIT = "pairs/s"


def reference_run(case="b20"):
    """One full run of the unmodified reference program; returns (seconds, pair interactions)."""
    exe = os.path.join(ROOT, "oracle", "_ref", "nbody")
    kind = "reference"
    if not os.path.exists(exe):  # the reference did not travel: fall back to the oracle port, and say so
        exe = os.path.join(ROOT, "oracle", "_build", "nbody_oracle")
        kind = "port"
    inp = os.path.join(CASES, case + ".in")
    out = "/tmp/bench_ref_%d.out" % os.getpid()
    t0 = time.perf_counter()
    subprocess.check_call([exe, inp, out] + (["200000", "0", "1"] if kind == "port" else []))
    dt = time.perf_counter() - t0
    lines = open(out).read().split("\n")
    gold = open(os.path.join(CASES, case + ".out")).read().split("\n")
    if lines[0] != gold[0] or lines[1] != gold[1]:
        raise RuntimeError("reference output differs from the golden")
    n = int(open(inp).readline().split()[0])
    hit = int(lines[1])
    steps = 200000 + (hit if hit >= 0 else 200000)  # Q1 runs all steps, Q2 stops at the hit (nbody.cc:114-138)
    if kind == "port":
        kats = json.load(open(os.path.join(ROOT, "tests", "golden", "oracle_kats.json")))[case]
        for d in kats["devices"]:  # the port also answers query 3 (forked at the reach step)
            end = d["q3_hit_step"] if d["q3_hit_step"] >= 0 else 200000
            if d["reach_step"] >= 0 and d["reach_step"] < hit:
                steps += end - d["reach_step"]
    return dt, steps * n * (n - 1), kind


SAMPLE_N = 8192  # bodies of the bounded CPU sample of the synthetic workload


def write_synthetic_input(path, n, seed=42):
    """The synthetic workload's generator parameters (SURVEY 8d C5: positions uniform in a 1e13 m cube centred at
    (-2.0e20, -2.9e20, 1.8e18), velocities N(0, 1e7 m/s), masses log-uniform in [1e20, 1e30] kg, body 0 planet, body 1
    asteroid, the last 4 bodies gravity devices) in the reference's input format (nbody.cc:22-39), pure Python: the
    reference arm loads nothing of this repo's."""
    import numpy as np

    rng = np.random.default_rng(seed)
    q = np.array([-2.0e20, -2.9e20, 1.8e18]) + (rng.random((n, 3)) - 0.5) * 1e13
    v = rng.normal(0.0, 1e7, (n, 3))
    m = 10.0 ** (20.0 + 10.0 * rng.random(n))
    with open(path, "w") as f:
        f.write("%d 0 1\n" % n)
        for i in range(n):
            f.write("%.17g %.17g %.17g %.17g %.17g %.17g %.17g %s\n" % (*q[i], *v[i], m[i], "device" if i >= n - 4 else "star"))


def reference_sample_run(n=SAMPLE_N, inp=None):
    """run_step of the reference on a bounded sample of the SAME workload (a synthetic system of the same generator
    parameters, n bodies): samples/nbody.cc with param::n_steps set to 1 at build time (oracle/Makefile pipes the
    source through sed; nothing else differs), i.e. two run_step calls (query 1 and query 2, nbody.cc:116,129).
    Returns (seconds, ordered pair interactions, kind)."""
    exe = os.path.join(ROOT, "oracle", "_ref", "nbody_steps1")
    kind = "reference"
    args = []
    if not os.path.exists(exe):
        exe, kind, args = os.path.join(ROOT, "oracle", "_build", "nbody_oracle"), "port", ["1", "0", "1"]
    own = inp is None
    if own:
        inp = "/tmp/bench_sample_%d_%d.in" % (n, os.getpid())
        write_synthetic_input(inp, n)
    out = "/tmp/bench_sample_%d.out" % os.getpid()
    t0 = time.perf_counter()
    subprocess.check_call([exe, inp, out] + args)
    dt = time.perf_counter() - t0
    if own:
        os.unlink(inp)
    return dt, 2 * n * (n - 1), kind


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    inp = "/tmp/bench_sample_%d_%d.in" % (SAMPLE_N, os.getpid())
    write_synthetic_input(inp, SAMPLE_N)
    for _ in range(args.warmup):
        reference_sample_run(inp=inp)
    tot_t, tot_p, kind = 0.0, 0, "reference"
    for _ in range(args.steps):
        dt, pairs, kind = reference_sample_run(inp=inp)
        tot_t += dt
        tot_p += pairs
    os.unlink(inp)
    val = tot_p / tot_t
    sample = ("per step: two run_step calls (query 1 + query 2, param::n_steps = 1 set at build time) of samples/nbody.cc, "
              "serial, on a %d-body synthetic system with the workload's generator parameters = %d ordered pairs; the "
              "full 65536-body step would take ~200 s on one core (pairs/s does not depend on n: same loop)"
              % (SAMPLE_N, 2 * SAMPLE_N * (SAMPLE_N - 1)))
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": tot_t / args.steps * 1e3, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "synthetic 65536-body single system", "reference_arm_sample_bodies": SAMPLE_N,
                   "same_config": "same workload and generator parameters, bounded to %d bodies per CPU step (see cpu_baseline.sample)" % SAMPLE_N},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": 1, "kind": kind, "sample": sample,
                         "host_cores_available": os.cpu_count()},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def init_nccl(dist, torch, dev):
    """init_process_group + the first collective with file descriptor 1 pointed at stderr: NCCL prints its version
    banner (NCCL_DEBUG=VERSION on these boxes) to stdout when the communicator is created, and stdout must carry the
    one JSON line only."""
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    try:
        dist.init_process_group("nccl", device_id=dev)
        dist.all_reduce(torch.zeros(1, device=dev))
        torch.cuda.synchronize(dev)
    finally:
        sys.stdout.flush()
        os.dup2(saved, 1)
        os.close(saved)


class ClockSampler:
    """SM clock, power and throttle reasons of one GPU sampled DURING the timed region: NVML from a thread every ~2 ms
    (a timed region can be as short as 10 ms at 8 GPUs), `nvidia-smi -lms 20` as the fallback."""
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
    MASKS = [0x8, 0x40, 0x20, 0x4]  # nvmlClocksThrottleReason{HwSlowdown, HwThermalSlowdown, SwThermalSlowdown, SwPowerCap}

    def __init__(self, uuid):
        self.proc, self.nvml, self.rows, self.lines, self.source = None, None, [], [], None
        self._stop = threading.Event()
        try:
            import pynvml

            pynvml.nvmlInit()
            try:
                self.h = pynvml.nvmlDeviceGetHandleByUUID(uuid.encode())
            except Exception:
                self.h = pynvml.nvmlDeviceGetHandleByUUID(uuid)
            self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.nvml, self.source = pynvml, "nvml, 2 ms"
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", uuid, "--query-gpu=" + self.FIELDS,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.source = "nvidia-smi -lms 20"
        except Exception:
            pass
        if self.proc:
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()

    def _poll(self):
        nv = self.nvml
        while not self._stop.is_set():
            try:
                ts = time.perf_counter()
                sm = float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                pw = nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0
                try:
                    rs = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                except Exception:
                    rs = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                self.rows.append((ts, sm, pw, rs))
            except Exception:
                pass
            time.sleep(0.002)

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append((time.perf_counter(), ln.strip()))

    def stop(self, t0, t1):
        sm, mx, pw, reasons = [], None, [], set()
        if self.nvml:
            self._stop.set()
            self.t.join(timeout=1.0)
            mx = self.mx
            for ts, s_, p_, rs in self.rows:
                if ts < t0 or ts > t1:
                    continue
                sm.append(s_)
                pw.append(p_)
                for nme, msk in zip(self.NAMES, self.MASKS):
                    if rs & msk:
                        reasons.add(nme)
        elif self.proc:
            time.sleep(0.15)
            self.proc.terminate()
            for ts, ln in self.lines:
                if ts < t0 or ts > t1 + 0.1:
                    continue
                f = [x.strip() for x in ln.split(",")]
                try:
                    sm.append(float(f[0]))
                    mx = float(f[1])
                    pw.append(float(f[2]))
                    for nme, val in zip(self.NAMES, f[3:7]):
                        if val.lower().startswith("active"):
                            reasons.add(nme)
                except Exception:
                    continue
        else:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no NVML, no nvidia-smi"]}
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons),
                "source": self.source}


DUMP_LIMIT_BYTES = 64 << 20


def dump_state(np, out_dir, q, v, n):
    """Planar q[3n] and v[3n] as returned by positions() / velocities(), saved as float64 [3, n] arrays.  Above
    DUMP_LIMIT_BYTES in all, the same fixed sample of bodies (seed 0, ascending index) is taken from both."""
    q, v = q.reshape(3, n), v.reshape(3, n)
    if q.nbytes + v.nbytes > DUMP_LIMIT_BYTES:
        keep = np.sort(np.random.default_rng(0).choice(n, DUMP_LIMIT_BYTES // (2 * 3 * 8), replace=False))
        q, v = q[:, keep], v[:, keep]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "positions.npy"), np.ascontiguousarray(q, dtype=np.float64))
    np.save(os.path.join(out_dir, "velocities.npy"), np.ascontiguousarray(v, dtype=np.float64))


def close_states(np, q, v, qo, vo):
    """FAST-math parity bar of SURVEY 8d C5: q within 1e-12*max|v|*dt (or 2 ulp), v within 1e-12 relative.
    Returns (ok, max relative v difference, max absolute q difference)."""
    dv = float(np.max(np.abs(v - vo) / np.maximum(np.abs(vo), 1e-300)))
    dq = float(np.abs(q - qo).max())
    ok = dq <= max(1e-12 * float(np.abs(vo).max()) * 60.0, 2 * float(np.spacing(np.abs(qo)).max())) and dv <= 1e-12
    return bool(ok), dv, dq


def make_system(nb, kind, system, rank, world, dev):
    if kind == "sym":
        return nb.SymShardedSystem(system, rank=rank, world=world, device=dev)
    if kind == "p2p":
        return nb.P2PShardedSystem(system, rank=rank, world=world, device=dev)
    return nb.ShardedSystem(system, rank=rank, world=world, device=dev)


def reference_gpu_block(nb):
    """BASELINE.md section 4 item 5 (opt-in, --reference-gpu): the reference's OWN GPU program, hw5.cu rebuilt for sm_100a
    (oracle/_ref/hw5_gpu, built from /root/reference by oracle/Makefile), as a process on b1024.  It hard-codes GPUs 0 and 1
    (hw5.cu:558-567), so it needs two visible GPUs.  Nothing of this repository is loaded by that process."""
    exe = os.path.join(ROOT, "oracle", "_ref", "hw5_gpu")
    if not os.path.exists(exe):
        return {"unavailable": "oracle/_ref/hw5_gpu was not built (reference tree or nvcc missing at build time)"}
    if nb.device_count() < 2:
        return {"unavailable": "needs two visible GPUs (hw5.cu:558-567 uses ordinals 0 and 1)"}
    inp, gold = os.path.join(CASES, "b1024.in"), open(os.path.join(CASES, "b1024.out"), "rb").read()
    out = "/tmp/bench_refgpu_%d.out" % os.getpid()
    t0 = time.perf_counter()
    try:
        r = subprocess.run([exe, inp, out], capture_output=True, timeout=600)
    except subprocess.TimeoutExpired:
        return {"wall_s": None, "timeout_s": 600}
    wall = time.perf_counter() - t0
    same = r.returncode == 0 and os.path.exists(out) and open(out, "rb").read() == gold
    return {"wall_s": wall, "rc": r.returncode, "byte_identical_to_golden": bool(same), "gpus": 2,
            "what": "process wall of the reference's hw5.cu (nvcc -std=c++11 -O3, -arch=sm_61 replaced by sm_100a) on b1024.in"}


def hw5_process_block(nb):
    """The real `hw5 <input> <output>` PROCESS on b1024 (BASELINE metric (i)) next to the floor of any CUDA process on
    this box (driver initialisation + one context + one empty kernel, tools/microbench/cuda_floor.cu)."""
    pkg = os.path.dirname(nb.LIB_PATH)
    exe, floor_exe = os.path.join(pkg, "hw5"), os.path.join(pkg, "cuda_floor")
    inp, gold = os.path.join(CASES, "b1024.in"), open(os.path.join(CASES, "b1024.out"), "rb").read()
    env = dict(os.environ, NB_VERBOSE="1")
    env.pop("CUDA_VISIBLE_DEVICES", None)  # the binary narrows it itself (to GPU 0)
    runs = []
    for rep in range(2):
        fl = None
        if os.path.exists(floor_exe):
            t0 = time.perf_counter()
            r = subprocess.run([floor_exe], capture_output=True, env=env, timeout=120)
            fl = {"wall_s": time.perf_counter() - t0}
            try:
                fl.update(json.loads(r.stdout.decode().strip().split("\n")[-1]))
            except Exception:
                pass
        out = "/tmp/bench_hw5_%d.out" % os.getpid()
        t0 = time.perf_counter()
        r = subprocess.run([exe, inp, out], capture_output=True, env=env, timeout=300)
        wall = time.perf_counter() - t0
        err = r.stderr.decode()
        laps = {}
        for ln in err.split("\n"):
            if "start-up (driver" in ln:
                laps["gpu_startup_s"] = float(ln.split()[-2])
            elif "three queries (nb_solve)" in ln:
                laps["solve_s"] = float(ln.split()[-2])
            elif "chain plan" in ln and "kernels" in ln:
                laps["kernels_s"] = float(ln.split("kernels")[-1].split()[0])
            elif "read input" in ln:
                laps["read_input_s"] = float(ln.split()[-2])
        same = r.returncode == 0 and os.path.exists(out) and open(out, "rb").read() == gold
        runs.append({"wall_s": wall, "rc": r.returncode, "byte_identical_to_golden": bool(same), "laps": laps, "cuda_floor": fl})
    best = min(runs, key=lambda x: x["wall_s"])
    return {"wall_s": best["wall_s"], "byte_identical_to_golden": all(x["byte_identical_to_golden"] for x in runs),
            "kernels_s": best["laps"].get("kernels_s"), "gpu_startup_s": best["laps"].get("gpu_startup_s"),
            "cuda_floor_s": best["cuda_floor"]["floor_s"] if best["cuda_floor"] and "floor_s" in best["cuda_floor"] else None,
            "runs": runs,
            "note": "process wall of the hw5 binary on one GPU (the CLI narrows CUDA_VISIBLE_DEVICES to GPU 0; the GPU is "
                    "started on a helper thread while the input is parsed); cuda_floor = wall of a CUDA process that only "
                    "initialises the driver, creates one context and launches one empty kernel on the same box: the part of "
                    "the wall no CUDA program can avoid here"}


def trev_equal(a, b):
    return (a.hit_step == b.hit_step and a.argmin_step == b.argmin_step and a.steps_done == b.steps_done
            and list(a.reach_step[:a.n_reach]) == list(b.reach_step[:b.n_reach]))


def ensemble_block(nb, np, torch, dist, rank, world, local, dev, steps, systems):
    """BASELINE config C4: `systems` independent 1024-body systems (member k = b1024.in with velocities scaled by
    1 + 1e-9 k), `steps` steps, split over the ranks with no collective."""
    base = nb.read_input(os.path.join(CASES, "b1024.in"))
    mine = list(range(rank, systems, world))
    S, n = len(mine), base.n
    q = np.tile(base.q, (S, 1))
    v = np.stack([base.v * (1 + 1e-9 * k) for k in mine])
    m = np.tile(base.m, (S, 1))
    isdev = np.tile(base.is_device, (S, 1))
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    ev, secs = nb.ensemble_run(q, v, m, isdev, [base.planet] * S, [base.asteroid] * S, kind=nb.KIND_Q2, step_end=steps, gpu=local)
    wall = time.perf_counter() - t0
    t = torch.tensor([secs, wall], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ok = None
    if rank == 0:  # member 0 is the golden system itself: its state must equal a plain trajectory's
        tr = nb.Trajectory(base, nb.KIND_Q2, gpu=local)
        tr_ev = tr.run(steps)
        qt = tr.state()[0]
        # the trajectory runs on the grid kernel (another summation order): positions within 2 ulp, same observers
        ok = bool((np.abs(qt - q[0]) <= 2 * np.spacing(np.abs(qt))).all() and trev_equal(tr_ev, ev[0]))
        tr.close()
    pairs = systems * steps * n * (n - 1)
    secs, wall = float(t[0]), float(t[1])
    return {"workload": "synthetic ensemble of %d independent 1024-body systems, %d steps (config C4)" % (systems, steps),
            "systems_per_rank": S, "gpu_s": secs, "wall_s_incl_copies": wall, "pairs_per_s": pairs / secs,
            "frac_of_fp64_peak": pairs / secs * PAIR_FLOPS / (world * FP64_PEAK_NOMINAL_TFLOPS * 1e12),
            "member0_equals_single_trajectory": ok,
            "member0_check": "positions within 2 ulp of, and observers equal to, the same system run as one trajectory on the grid kernel",
            "kernel": "traj_sym_kernel (one block per system, all steps in one launch; every unordered pair of different 128-body groups evaluated once)"}


def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    nb = importlib.import_module(PKG)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available() or nb.device_count() < 1:
        raise SystemExit("bench.py needs a CUDA device: the hot path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        init_nccl(dist, torch, dev)
    if world != args.gpus and rank == 0:
        print("warning: --gpus %d but WORLD_SIZE %d" % (args.gpus, world), file=sys.stderr)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    n = args.n
    system = nb.synthetic_system(n, seed=42)
    sh = make_system(nb, args.exchange, system, rank, world, dev)
    exchange_bytes = sh.bytes_exchanged_per_step()
    flush = None if args.no_l2_flush else torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    uuid = str(torch.cuda.get_device_properties(dev).uuid)
    uuid = uuid if uuid.startswith("GPU-") else "GPU-" + uuid

    # ---- device-resident measurement ---------------------------------------------------------------
    sampler = ClockSampler(uuid) if rank == 0 else None
    t_warm = time.perf_counter()
    for _ in range(args.warmup):
        sh.advance(1)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    launches0 = nb.kernel_launches()
    t0 = time.perf_counter()
    for k in range(args.steps):
        if flush is not None:
            flush.zero_()
        ev[k][0].record()
        sh.advance(1)
        ev[k][1].record()
    barrier()
    t1 = time.perf_counter()
    launches = nb.kernel_launches() - launches0
    dev_ms = sum(a.elapsed_time(b) for a, b in ev)
    dev_ms = max_over_ranks(dev_ms)
    pairs_per_step = n * (n - 1)
    value = pairs_per_step * args.steps / (dev_ms * 1e-3)
    if args.dump_outputs:
        q_out, v_out = sh.positions(), sh.velocities()  # every rank: velocities() gathers the shards
        if rank == 0:
            dump_state(np, args.dump_outputs, q_out, v_out, n)

    # ---- the acceleration kernel alone (roofline) ---------------------------------------------------
    nb.profile_enable(True)
    for _ in range(min(args.steps, 10)):
        if flush is not None:
            flush.zero_()
        sh.advance(1)
    torch.cuda.synchronize()
    accel_ms, accel_n = nb.profile_read()
    nb.profile_enable(False)
    accel_ms = max_over_ranks(accel_ms / max(accel_n, 1))
    if args.exchange == "sym":
        # ordered pairs one launch of this rank covers (2 x its unordered pairs + the one-sided diagonal rows, self pairs excluded)
        rank_pairs = sh.pairs_per_step() - sh.i_count
        kernel, instr_per_pair = "sym_accel_kernel", 10
    else:
        rank_pairs = sh.i_count * (n - 1)
        kernel, instr_per_pair = "large_accel_kernel", 16
    flops_per_launch = PAIR_FLOPS * rank_pairs
    achieved = flops_per_launch / (accel_ms * 1e-3) / 1e12
    peak_measured = nb.fp64_peak(local)
    traffic, traffic_src = None, None
    tfile = os.path.join(ROOT, "profiles", "r02_sym_accel_traffic.json")
    if n == 65536 and world == 1 and args.exchange == "sym" and os.path.exists(tfile):
        tj = json.load(open(tfile))
        traffic, traffic_src = tj["dram_bytes_per_launch"], tj["source"]

    # ---- end to end through the host-buffer operator (same kernels, same exchange as `value`) --------
    ib, ic = sh.i_begin, sh.i_count
    qh = torch.from_numpy(system.q.reshape(3, n)[:, ib:ib + ic].copy()).pin_memory()
    vh = torch.from_numpy(system.v.reshape(3, n)[:, ib:ib + ic].copy()).pin_memory()
    e2e_sys = make_system(nb, args.exchange, system, rank, world, dev)
    if args.exchange != "sym":  # the row-kernel drivers take all positions from the host
        qh = torch.from_numpy(system.q.copy()).pin_memory()
    for _ in range(args.warmup):
        h2d, d2h = e2e_sys.step_host(qh, vh)
    barrier()
    te0 = time.perf_counter()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        h2d, d2h = e2e_sys.step_host(qh, vh)
    e1.record()
    barrier()
    e2e_wall = max_over_ranks(time.perf_counter() - te0)
    e2e_ms = max_over_ranks(e0.elapsed_time(e1))
    e2e_value = pairs_per_step * args.steps / max(e2e_ms * 1e-3, e2e_wall if world == 1 else 0.0)
    e2e_q_own = qh.numpy().copy() if args.exchange == "sym" else None
    clocks = None
    if sampler:
        # a timed region shorter than ~0.2 s (8 GPUs: 20 steps = 9 ms) holds too few samples: widen the window to everything
        # from the warm-up to the end of the e2e loop - the same kernels on the same GPU throughout
        short = (t1 - t0) < 0.2
        clocks = sampler.stop(t_warm if short else t0, time.perf_counter() if short else t1)
        clocks["window"] = "warm-up + timed + roofline + e2e loops" if short else "timed"
    launches_total = nb.kernel_launches()

    # ---- parity of exactly what was timed (outside the timed regions) -------------------------------
    parity = None
    if not args.no_parity:
        K = 3
        a = make_system(nb, args.exchange, system, rank, world, dev)
        a.advance(K)
        qa, va = a.positions(), a.velocities()
        b = make_system(nb, args.exchange, system, rank, world, dev)
        b.advance(K)
        qb, vb = b.positions(), b.velocities()
        deterministic = bool(np.array_equal(qa, qb) and np.array_equal(va, vb))
        c = nb.ShardedSystem(system, rank=rank, world=world, device=dev)  # row kernel + NCCL all-gather: independent path
        c.advance(K)
        torch.cuda.synchronize()
        qc, vc = c.positions(), c.velocities()
        ok_row, dv_row, dq_row = close_states(np, qa, va, qc, vc)
        q1, v1 = system.q.copy(), system.v.copy()
        nb.run_steps(0, K, n, q1, v1, system.m, system.is_device, gpu=local)  # one rank, one GPU, host-buffer operator
        ok_one, dv_one, dq_one = close_states(np, qa, va, q1, v1)
        # the e2e arm advanced warmup + steps steps from the same seed state through host buffers: same state as the
        # resident arm after as many steps
        e2e_ok = None
        if e2e_q_own is not None:
            d = make_system(nb, args.exchange, system, rank, world, dev)
            d.advance(args.warmup + args.steps)
            qd = d.positions().reshape(3, n)[:, ib:ib + ic]
            e2e_ok = bool(np.array_equal(qd, e2e_q_own))
            d.close() if hasattr(d, "close") else None
        flags = torch.tensor([deterministic, ok_row, ok_one, 1 if e2e_ok in (None, True) else 0], dtype=torch.int32, device=dev)
        if world > 1:
            dist.all_reduce(flags, op=dist.ReduceOp.MIN)
        parity = {"steps": K, "run_to_run_bit_identical": bool(flags[0]), "vs_row_kernel_nccl_path": bool(flags[1]),
                  "vs_row_kernel_max_rel_dv": dv_row, "vs_one_rank_run_steps": bool(flags[2]), "vs_one_rank_max_rel_dv": dv_one,
                  "vs_one_rank_bit_identical": bool(np.array_equal(qa, q1) and np.array_equal(va, v1)),
                  "e2e_state_equals_resident_state": bool(flags[3]), "exchange_status_word": 0,
                  "tolerance": "v within 1e-12 relative, q within max(1e-12*max|v|*dt, 2 ulp) (SURVEY 8d C5); positions() raises if a peer wait timed out",
                  "all_ranks": True}
        if world == 1 and args.exchange == "sym":
            emu = {}
            for w in (2, 8):
                lw = nb.SymLocalWorld(system, w, device=dev)
                lw.advance(K)
                okw, dvw, _ = close_states(np, lw.positions(), lw.velocities(), qa, va)
                lw.close()
                emu["world_%d" % w] = {"ok": okw, "max_rel_dv": dvw}
            parity["multi_rank_path_emulated_on_this_gpu"] = emu
        for x in (a, b):
            x.close() if hasattr(x, "close") else None
    for x in (sh, e2e_sys):
        x.close() if hasattr(x, "close") else None

    # ---- b1024 three-query end to end (the other half of the BASELINE metric) -----------------------
    b1024 = None
    if not args.no_b1024:
        s1024 = nb.read_input(os.path.join(CASES, "b1024.in"))
        barrier()
        tb = time.perf_counter()
        ans, gsecs, pairs = nb.solve_distributed(s1024, rank, world, local)
        barrier()
        wall = max_over_ranks(time.perf_counter() - tb)
        text = nb.format_output(ans.min_dist, ans.hit_time_step, ans.gravity_device_id, ans.missile_cost)
        gold = open(os.path.join(CASES, "b1024.out")).read()
        gl, tl = gold.split("\n"), text.split("\n")
        ok = tl[1] == gl[1] and tl[2] == gl[2] and abs(float(tl[0]) - float(gl[0])) <= 1e-6 * float(gl[0])
        b1024 = {"solve_wall_s": wall, "gpu_s": gsecs, "pairs_per_s_gpu": pairs / gsecs if gsecs else None,
                 "trajectories": ans.n_trajectories, "matches_golden": bool(ok), "line1_byte_identical": tl[0] == gl[0],
                 "us_per_step_q1": None,
                 "note": "in-process solve (contexts already created); as many GPUs as trajectories: Q1, Q2 and one Q3 trajectory per device from step 0, one per rank; fewer: Q1 on rank 0, Q2 -> Q3 candidates forked from Q2 on rank 1 (chain plan, nb_host.cu)"}
        if rank == 0:
            # step latency of ONE system spread over the GPU (the quantity that bounds the >= 4-GPU solve): query 1, all steps
            tr = nb.Trajectory(s1024, nb.KIND_Q1, gpu=local)
            tr.run(2000)
            tq = time.perf_counter()
            tr.run(nb.N_STEPS)
            b1024["us_per_step_q1"] = (time.perf_counter() - tq) / (nb.N_STEPS - 2000) * 1e6
            tr.close()
            b1024["torn_records_detected"] = nb.grid_torn_records()
        if rank == 0 and not args.no_hw5_process:
            b1024["hw5_process"] = hw5_process_block(nb)
        if rank == 0 and args.reference_gpu:
            b1024["reference_hw5_cu_process"] = reference_gpu_block(nb)
        barrier()

    # ---- config C4: the synthetic ensemble ----------------------------------------------------------
    ensemble = None
    if not args.no_ensemble:
        ensemble = ensemble_block(nb, np, torch, dist, rank, world, local, dev, args.ensemble_steps, args.systems)

    # ---- CPU baselines on this box's host cores (N = 1 only) ----------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        dt, pairs, kind = reference_sample_run()
        cpu = {"value": pairs / dt, "unit": UNIT, "cores": 1, "kind": kind, "seconds": dt,
               "sample": "two run_step calls (param::n_steps = 1 set at build time) of samples/nbody.cc, serial, on a %d-body "
                         "synthetic system with the workload's generator parameters (%d ordered pairs)" % (SAMPLE_N, pairs),
               "host_cores_available": os.cpu_count(), "extras": cpu_extras(nb, np, system, args)}

    if rank == 0:
        exch = {"sym": "symmetric stepper: partial accelerations and pos4 rows stored straight into the owners' / every rank's memory "
                       "(peer-mapped buffers), in-kernel arrival waits, 2 launches per step, no NCCL on the data path",
                "p2p": "row kernel, P2P stores fused into the integrate kernel (peer-mapped buffers, no NCCL on the data path)",
                "nccl": "row kernel, in-place NCCL all-gather of pos4 rows"}[args.exchange]
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dev_ms / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "synthetic 65536-body single system" if n == 65536 else "synthetic %d-body single system" % n,
                       "n_bodies": n, "seed": 42, "bodies_per_rank": sh.i_count, "pairs_per_step": pairs_per_step,
                       "math": "fast; every unordered pair evaluated once, both accelerations accumulated (10 FP64 instr per ordered pair)"
                               if args.exchange == "sym" else "fast (16 FP64 instr per ordered pair)",
                       "parallelism": "body-sharded x%d" % world, "exchange": exch if world > 1 else "none (1 GPU)",
                       "l2": "not flushed" if flush is None else "flushed between timed steps (256 MiB memset, outside the per-step events)",
                       "exchange_bytes_per_rank_per_step": exchange_bytes},
            "frac_of_fp64_peak": value * PAIR_FLOPS / (world * FP64_PEAK_NOMINAL_TFLOPS * 1e12),
            "roofline": {"bound": "fp64", "achieved": achieved, "peak": FP64_PEAK_NOMINAL_TFLOPS, "unit": "TFLOP/s",
                         "frac": achieved / FP64_PEAK_NOMINAL_TFLOPS,
                         "traffic": traffic, "traffic_source": traffic_src,
                         "kernel": kernel, "kernel_ms": accel_ms,
                         "peak_source": "nominal 148 SM x 64 FMA/clk x 2 x 1.965 GHz (MEASURED_PEAKS.json has no FP64 entry)",
                         "peak_measured_dfma": peak_measured, "frac_of_measured": achieved / peak_measured,
                         "flops_per_pair": PAIR_FLOPS, "fp64_instr_per_pair": instr_per_pair,
                         "ordered_pairs_per_launch": rank_pairs,
                         "note": "compute-bound path: algorithmic bytes are 104 B x n per step (intensity ~12600 flop/B), "
                                 "so the roofline is the FP64 pipe, not HBM or tensor cores (SURVEY.md 8d); achieved = 20 flop x "
                                 "ordered pairs per launch / CUDA-event duration of the kernel"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": e2e_ms / args.steps,
                    "note": "per rank per step: this rank's positions and velocities host -> device (pinned), published to every "
                            "rank, the step's kernels, the new rows device -> host; same kernels and exchange as `value`"},
            "gpu_launches": launches,
            "gpu_launches_total_process": launches_total,
            "clocks": clocks,
            "parity": parity,
            "cpu_baseline": cpu,
            "b1024": b1024,
            "ensemble": ensemble,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def cpu_extras(nb, np, system, args):
    """BASELINE.md section 4 items 2-4, each bounded."""
    ex = {}
    try:
        dt, pairs, kind = reference_run("b20")
        ex["b20_full"] = {"seconds": dt, "pairs_per_s": pairs / dt, "cores": 1, "kind": kind,
                          "what": "full b20.in run of the unmodified samples/nbody.cc (query 1 + query 2), output lines 1-2 equal the golden"}
    except Exception as e:  # noqa: BLE001
        ex["b20_full"] = {"error": str(e)}
    if getattr(args, "cpu_b100_full", False):  # BASELINE.md section 4 item 2: about three minutes of one host core, opt-in
        try:
            dt, pairs, kind = reference_run("b100")
            ex["b100_full"] = {"seconds": dt, "pairs_per_s": pairs / dt, "cores": 1, "kind": kind,
                               "what": "full b100.in run of the unmodified samples/nbody.cc (query 1 + query 2), output lines 1-2 equal the golden"}
        except Exception as e:  # noqa: BLE001
            ex["b100_full"] = {"error": str(e)}
    exe = os.path.join(ROOT, "oracle", "_ref", "nbody_steps200")
    if os.path.exists(exe):
        out = "/tmp/bench_w200_%d.out" % os.getpid()
        t0 = time.perf_counter()
        subprocess.check_call([exe, os.path.join(CASES, "b1024.in"), out])
        dt = time.perf_counter() - t0
        pairs = 2 * 200 * 1024 * 1023  # query 1 and query 2, 200 steps each (no hit that early)
        full_pairs = (200000 + 148198) * 1024 * 1023  # nbody.cc runs Q1 to the end and Q2 to the hit step (golden: 148198)
        ex["b1024_window_200_steps"] = {"seconds": dt, "pairs_per_s": pairs / dt, "cores": 1, "kind": "reference",
                                        "extrapolated_full_b1024_q1_q2_seconds": full_pairs / (pairs / dt),
                                        "what": "samples/nbody.cc with param::n_steps = 200 (set at build time) on b1024.in; the full "
                                                "Q1 + Q2 run is EXTRAPOLATED linearly from this window"}
    # the repo's CPU oracle (OpenMP over i, bit-identical to serial) on all host cores: one step of the 65536-body system,
    # which is also the full-size parity check of the GPU step
    try:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import oracle_binding as orc

        n = system.n
        cores = os.cpu_count()
        if cores >= 16 and not args.no_oracle_full_step:
            qo, vo = system.q.copy(), system.v.copy()
            t0 = time.perf_counter()
            orc.run_steps(orc.MODE_SQRT3, n, qo, vo, system.m, system.is_device, 0, 1, nthreads=cores)
            dt = time.perf_counter() - t0
            q, v = system.q.copy(), system.v.copy()
            nb.run_steps(0, 1, n, q, v, system.m, system.is_device, gpu=0)
            ok, dv, dq = close_states(np, q, v, qo, vo)
            ex["openmp_oracle_65536_one_step"] = {"seconds": dt, "pairs_per_s": n * (n - 1) / dt, "cores": cores, "kind": "port",
                                                  "gpu_step_matches": ok, "max_rel_dv": dv, "max_abs_dq_m": dq,
                                                  "what": "oracle/nbody_oracle.cc, sqrt(r2^3) mode, OpenMP over i on all host cores"}
        else:
            ns = 16384
            sub = nb.synthetic_system(ns, seed=42)
            qo, vo = sub.q.copy(), sub.v.copy()
            t0 = time.perf_counter()
            orc.run_steps(orc.MODE_SQRT3, ns, qo, vo, sub.m, sub.is_device, 0, 1, nthreads=cores)
            dt = time.perf_counter() - t0
            ex["openmp_oracle_16384_one_step"] = {"seconds": dt, "pairs_per_s": ns * (ns - 1) / dt, "cores": cores, "kind": "port",
                                                  "what": "fewer than 16 host cores: one step of a 16384-body system instead of 65536"}
    except Exception as e:  # noqa: BLE001
        ex["openmp_oracle"] = {"error": str(e)}
    return ex


def run_ensemble(args):
    """BASELINE config 4: 1024 independent 1024-body systems (member k = b1024.in with velocities scaled by
    1 + 1e-9 k, SURVEY 8d C4), split over the ranks with no collective; one block per system, one launch."""
    import numpy as np
    import torch
    import torch.distributed as dist

    nb = importlib.import_module(PKG)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        init_nccl(dist, torch, dev)
    S_total = args.systems
    base = nb.read_input(os.path.join(CASES, "b1024.in"))
    mine = list(range(rank, S_total, world))
    S, n = len(mine), base.n
    q0 = np.tile(base.q, (S, 1))
    v0 = np.stack([base.v * (1 + 1e-9 * k) for k in mine])
    m = np.tile(base.m, (S, 1))
    isdev = np.tile(base.is_device, (S, 1))
    pl, ast = [base.planet] * S, [base.asteroid] * S

    def once(steps):
        q, v = q0.copy(), v0.copy()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        ev, secs = nb.ensemble_run(q, v, m, isdev, pl, ast, kind=nb.KIND_Q2, step_end=steps, gpu=local)
        wall = time.perf_counter() - t0
        t = torch.tensor([secs, wall], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0]), float(t[1]), ev, q

    once(max(args.warmup, 1))
    uuid = str(torch.cuda.get_device_properties(dev).uuid)
    sampler = ClockSampler(uuid if uuid.startswith("GPU-") else "GPU-" + uuid) if rank == 0 else None
    ts0 = time.perf_counter()
    secs, wall, ev, q = once(args.steps)
    clocks = sampler.stop(ts0, time.perf_counter()) if sampler else None
    # member 0 of rank 0 is the golden system itself: its state must equal a plain trajectory's
    ok = True
    if rank == 0:
        t = nb.Trajectory(base, nb.KIND_Q2, gpu=local)
        tev = t.run(args.steps)
        qt = t.state()[0]
        ok = bool((np.abs(qt - q[0]) <= 2 * np.spacing(np.abs(qt))).all() and trev_equal(tev, ev[0]))
    pairs = S_total * args.steps * n * (n - 1)
    if rank == 0:
        print(json.dumps({
            "metric": METRIC, "value": pairs / secs, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 1), "ms_per_step": secs / args.steps * 1e3, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic (b1024.in with scaled velocities)",
            "config": {"workload": "synthetic ensemble of %d independent 1024-body systems" % S_total,
                       "systems_per_rank": S, "parallelism": "ensemble x%d, no collective" % world,
                       "kernel": "traj_sym_kernel (one block per system, whole run in one launch)"},
            "frac_of_fp64_peak": pairs / secs * PAIR_FLOPS / (world * FP64_PEAK_NOMINAL_TFLOPS * 1e12),
            "e2e": {"value": pairs / wall, "unit": UNIT, "h2d_bytes_per_step": int(S * n * 57 / args.steps),
                    "d2h_bytes_per_step": int(S * n * 48 / args.steps), "note": "states uploaded once per launch, not per step"},
            "roofline": {"bound": "fp64", "achieved": pairs / secs * PAIR_FLOPS / 1e12 / world, "peak": FP64_PEAK_NOMINAL_TFLOPS,
                         "unit": "TFLOP/s", "frac": pairs / secs * PAIR_FLOPS / (world * FP64_PEAK_NOMINAL_TFLOPS * 1e12),
                         "traffic": None, "kernel": "traj_sym_kernel", "note": "per GPU; the whole launch is this kernel"},
            "clocks": clocks, "member0_equals_single_trajectory": ok, "gpu_launches": 2}), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--n", type=int, default=65536)
    ap.add_argument("--no-b1024", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-l2-flush", action="store_true")
    ap.add_argument("--workload", default="large", choices=["large", "ensemble"])
    ap.add_argument("--exchange", default=os.environ.get("NB_EXCHANGE", "sym"), choices=["sym", "nccl", "p2p"])
    ap.add_argument("--systems", type=int, default=1024)
    ap.add_argument("--ensemble-steps", type=int, default=10000)
    ap.add_argument("--no-ensemble", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-hw5-process", action="store_true")
    ap.add_argument("--no-oracle-full-step", action="store_true")
    ap.add_argument("--reference-gpu", action="store_true",
                    help="also run the reference's own hw5.cu (rebuilt for sm_100a, needs two visible GPUs) on b1024 as a process")
    ap.add_argument("--cpu-b100-full", action="store_true",
                    help="also time the full b100 run of the unmodified samples/nbody.cc (about 3 minutes of one host core)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps of the large workload, write the state they computed to DIR as positions.npy "
                         "and velocities.npy (float64, planar [3, n]; a fixed sample of bodies above 64 MiB in all)")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 0)
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload != "large"):
        ap.error("--dump-outputs applies to the large workload of --impl ours")
    if args.impl == "reference":
        run_reference_arm(args)
    elif args.workload == "ensemble":
        run_ensemble(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
