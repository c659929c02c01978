"""Kernel time of the diagnostics (nb_diagnostics: sym_potential_kernel + sym_diag_sum_kernel) for two shapes:
one system of 65 536 bodies, and config C4's shape, 1 024 systems of 1 024 bodies.

For each shape: REPS warmed calls; the time is the call's gpu_seconds (CUDA events around the two kernels, copies
excluded).  Reported: median and min, unordered pairs per second (n(n-1)/2 per system), and the share of the FP64 rate
nb_fp64_peak measures in this process, at 12 FP64 instructions per unordered pair (11 in pair_rinv, one accumulate FMA;
nb_fp64_peak counts a DFMA as two flops).  For comparison, the time per step of nb_run_steps (the symmetric stepper) at
65 536 bodies, host clock around a 40-step call that ends in a synchronise.  One JSON line per result, the card's name
and power limit first.

    python tools/diag_bench.py
"""
import importlib
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
nb = importlib.import_module("nthu_ipc_nbody-simulation_b200")

REPS = 20
FP64_PER_PAIR = 12


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    f = (r.stdout.strip().split(", ") + ["?", "?"])[:3] if r.returncode == 0 else ("?", "?", "?")
    return dict(card=f[0], power_limit=f[1], max_sm_clock=f[2])


def measure(label, S, n, peak_tflops):
    base = nb.generate_system(n, seed=42)
    q = np.tile(base.q, (S, 1))
    v = np.stack([base.v * (1.0 + 1e-9 * k) for k in range(S)])
    m, dev = np.tile(base.m, (S, 1)), np.tile(base.is_device, (S, 1))
    for _ in range(3):
        nb.diagnostics(q, v, m, dev, step=1000, return_seconds=True)
    secs = [nb.diagnostics(q, v, m, dev, step=1000, return_seconds=True)[1] for _ in range(REPS)]
    t = statistics.median(secs)
    pairs = S * n * (n - 1) / 2
    tiles = -(-n // nb.DIAG_TILE)
    evaluated = S * tiles * (tiles + 1) / 2 * nb.DIAG_TILE ** 2
    share = pairs * FP64_PER_PAIR / (peak_tflops * 1e12 / 2) / t
    return dict(shape=label, systems=S, n=n, reps=REPS, kernel_ms_median=1e3 * t, kernel_ms_min=1e3 * min(secs),
                unordered_pairs=pairs, pairs_evaluated_in_tiles=evaluated, pairs_per_s=pairs / t,
                fp64_peak_tflops=peak_tflops, share_of_fp64_peak=share, samples_ms=[1e3 * x for x in secs])


def step_time(n=65536, steps=40):
    s = nb.generate_system(n, seed=42)
    q, v = s.q.copy(), s.v.copy()
    nb.run_steps(0, 2, n, q, v, s.m, s.is_device)  # warm-up
    t0 = time.perf_counter()
    nb.run_steps(2, 2 + steps, n, q, v, s.m, s.is_device)
    return dict(shape="nb_run_steps, one system", n=n, steps=steps, ms_per_step=1e3 * (time.perf_counter() - t0) / steps)


def main():
    print(json.dumps(card()), flush=True)
    peak = nb.fp64_peak(0)
    print(json.dumps(dict(fp64_peak_tflops=peak)), flush=True)
    print(json.dumps(measure("one system of 65536 bodies", 1, 65536, peak)), flush=True)
    print(json.dumps(measure("config C4: 1024 systems of 1024 bodies", 1024, 1024, peak)), flush=True)
    print(json.dumps(step_time()), flush=True)


if __name__ == "__main__":
    main()
