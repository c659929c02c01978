"""Throughput of nb_ensemble_run above 1024 bodies (nb_ens.cu) against the sequential path.

For each (S, n): S generated systems (nb.generate_system, PLAIN kind, FAST math) advanced together by nb_ensemble_run,
enough steps for at least ~1 s of kernels; ordered pairs/s = S n (n - 1) steps / gpu_seconds (CUDA events around the
call's kernels, pack and unpack included).  The baseline is nb_run_steps on one member of the same size (one system per
call, the symmetric stepper), timed with a host clock around the call, which ends in a device synchronise and so includes
its allocation and copies; it runs enough steps for ~1 s too.  The two alternate, REPS times each, in this one process.
Rates are compared with the nominal 1.86e12 pairs/s (37.2 TFLOP/s at 20 FP64 flop per ordered pair) and with
nb_fp64_peak measured in the same process.  One JSON line per result, the card's name and power limit first.

    python tools/large_ensemble_bench.py [S:n ...]
"""
import importlib
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
nb = importlib.import_module("nthu_ipc_nbody-simulation_b200")

REPS = 3
WORKLOADS = [(512, 1025), (256, 2048), (64, 4096), (16, 8192), (4, 16384), (2, 65536)]
NOMINAL_PAIRS = 37.2e12 / 20  # ordered pairs/s at the nominal FP64 rate, 20 flop per pair
TARGET_S = 1.0


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    name, power = (r.stdout.strip().split(", ") + ["?"])[:2] if r.returncode == 0 else ("?", "?")
    return dict(card=name, power_limit=power)


def ensemble(systems, steps):
    import numpy as np

    q = np.stack([s.q for s in systems])
    v = np.stack([s.v for s in systems])
    m = np.stack([s.m for s in systems])
    dev = np.stack([s.is_device for s in systems])
    _, secs = nb.ensemble_run(q, v, m, dev, [s.planet for s in systems], [s.asteroid for s in systems], step_end=steps)
    return secs


def sequential(s, steps):
    q, v = s.q.copy(), s.v.copy()
    t = time.perf_counter()
    nb.run_steps(0, steps, s.n, q, v, s.m, s.is_device)
    return time.perf_counter() - t


def measure(S, n, peak_pairs):
    systems = [nb.generate_system(n, seed=k) for k in range(S)]
    pairs_step = S * n * (n - 1)
    # steps for ~TARGET_S of kernels, from a short run of each path
    ens_steps = max(20, int(TARGET_S * 5 / ensemble(systems, 5) + 0.5))
    per_step = sequential(systems[0], 20) / 20
    seq_steps = max(20, int(TARGET_S / per_step + 0.5))
    ens, seq = [], []
    for _ in range(REPS):
        ens.append(pairs_step * ens_steps / ensemble(systems, ens_steps))
        seq.append(n * (n - 1) * seq_steps / sequential(systems[0], seq_steps))
    e, s = statistics.median(ens), statistics.median(seq)
    return dict(S=S, n=n, steps=ens_steps, pairs_per_s=e, of_nominal=e / NOMINAL_PAIRS, of_measured_peak=e / peak_pairs,
                sequential_steps=seq_steps, sequential_pairs_per_s=s, speedup=e / s, samples=ens, sequential_samples=seq)


def main():
    print(json.dumps(card()), flush=True)
    peak = nb.fp64_peak(0)
    peak_pairs = peak * 1e12 / 20
    print(json.dumps(dict(fp64_peak_tflops=peak, peak_pairs_per_s=peak_pairs)), flush=True)
    loads = [tuple(int(x) for x in a.split(":")) for a in sys.argv[1:]] or WORKLOADS
    for S, n in loads:
        print(json.dumps(measure(S, n, peak_pairs)), flush=True)


if __name__ == "__main__":
    main()
