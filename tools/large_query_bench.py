"""Cost of the per-step observer on the large-N query path (n > 1024).

For each n, on a generated system (nb.generate_system) whose Q2 does not hit within the steps run: microseconds per
trajectory step of solve_partial with one part (the chain plan: Q1 and Q2, stepped one after the other, each step followed
by large_observe_kernel) against nb_run_steps (the same steppers, no observer) at the same n and step count.  The two
alternate, REPS times each, in this one process; the table gives the median of each and their ratio.  Then the wall time
of the hw5 binary on b1024 padded with massless probes to 2048 bodies.  Times are host clocks around calls that end in a
device synchronise, so they include each call's set-up (allocation, upload, stepper handle).  One JSON line per result,
the card's name and power limit first.

    python tools/large_query_bench.py [n ...]
"""
import importlib
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
nb = importlib.import_module("nthu_ipc_nbody-simulation_b200")

REPS = 3
SIZES = [1025, 2048, 4096, 16384, 65536]


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    name, power = (r.stdout.strip().split(", ") + ["?"])[:2] if r.returncode == 0 else ("?", "?")
    return dict(card=name, power_limit=power)


def steps_for(n):
    """At least ~1 s of stepping per run_steps call: 2.95 ms per step at 65 536 bodies, scaled by n^2, and no less than
    20 us per step below ~4 096 bodies, where a step is launch-bound."""
    per_step = max(20e-6, 2.95e-3 * (n / 65536) ** 2)
    return max(100, int(1.0 / per_step + 0.5))


def timed(f):
    t = time.perf_counter()
    out = f()
    return time.perf_counter() - t, out


def measure(n):
    s = nb.generate_system(n, seed=7)
    steps = steps_for(n)

    def q2():
        evs, _, pairs = nb.solve_partial(s, 0, 0, 1, n_steps=steps)
        return evs, pairs // (n * (n - 1))

    def plain():
        q, v = s.q.copy(), s.v.copy()
        nb.run_steps(0, steps, n, q, v, s.m, s.is_device)

    timed(q2), timed(plain)  # warm-up: module load, tables, stepper handle
    tq, tp = [], []
    for _ in range(REPS):
        dt, (evs, traj_steps) = timed(q2)
        tq.append(dt / traj_steps)
        tp.append(timed(plain)[0] / steps)
    us_q, us_p = 1e6 * statistics.median(tq), 1e6 * statistics.median(tp)
    return dict(n=n, steps=steps, q2_hit_step=evs[1].hit_step, trajectory_steps=traj_steps, us_per_step_query=us_q,
                us_per_step_run_steps=us_p, ratio=us_q / us_p, query_samples_us=[1e6 * x for x in tq],
                run_steps_samples_us=[1e6 * x for x in tp])


def hw5_padded_b1024():
    from test_gpu_large_queries import padded

    with tempfile.TemporaryDirectory() as d:
        inp, out = os.path.join(d, "in"), os.path.join(d, "out")
        nb.write_input(inp, padded(nb, "b1024", 2048))
        walls = []
        for _ in range(REPS):
            dt, r = timed(lambda: subprocess.run([nb.HW5_PATH, inp, out], capture_output=True, text=True))
            if r.returncode:
                raise SystemExit(r.stderr)
            walls.append(dt)
        lines = open(out).read().split("\n")[:3]
    return dict(case="b1024 padded to 2048 bodies", hw5_wall_s=walls, output=lines)


def main():
    print(json.dumps(card()), flush=True)
    for n in [int(a) for a in sys.argv[1:]] or SIZES:
        print(json.dumps(measure(n)), flush=True)
    print(json.dumps(hw5_padded_b1024()), flush=True)


if __name__ == "__main__":
    main()
