"""Quick on-box timing probe (not the bench): python tools/probe.py <what> [args]."""
import importlib
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
nb = importlib.import_module("nthu_ipc_nbody-simulation_b200")
G = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "testcases")


def peak():
    print("fp64 peak TF/s:", nb.fp64_peak(0), flush=True)


def peakv():
    for v in (0, 1, 2):
        print("fp64 peak variant %d (0: reg*UR+reg.reuse, 1: 3 distinct regs, 2: shared multiplicand): %.2f TF/s" % (v, nb.fp64_peak(0, v)), flush=True)


def traj(case="b1024", steps=2000):
    s = nb.read_input(os.path.join(G, case + ".in"))
    steps = int(steps)
    for kind in (nb.KIND_Q1,):
        t = nb.Trajectory(s, kind)
        t.run(10)
        t0 = time.time()
        t.run(10 + steps)
        dt = time.time() - t0
        print("%s single trajectory: %.2f us/step, %.3e pairs/s" % (case, dt / steps * 1e6, s.n * (s.n - 1) * steps / dt), flush=True)
        t.close()


def trajrep(case="b1024", steps=100000, reps=6):
    """Step latency of one trajectory, repeated (fresh trajectory each time): run-to-run spread of the grid kernel."""
    s = nb.read_input(os.path.join(G, case + ".in"))
    steps, out = int(steps), []
    for _ in range(int(reps)):
        t = nb.Trajectory(s, nb.KIND_Q1)
        t.run(10)
        t0 = time.time()
        t.run(10 + steps)
        out.append((time.time() - t0) / steps * 1e6)
        t.close()
    print("%s us/step over %d reps of %d steps: %s | min %.2f max %.2f" % (case, len(out), steps, " ".join("%.2f" % x for x in out), min(out), max(out)), flush=True)


def ens(S=148, steps=300, case="b1024"):
    S, steps = int(S), int(steps)
    s = nb.read_input(os.path.join(G, case + ".in"))
    q = np.tile(s.q, (S, 1))
    v = np.stack([s.v * (1 + 1e-9 * k) for k in range(S)])
    m = np.tile(s.m, (S, 1))
    dev = np.tile(s.is_device, (S, 1))
    nb.ensemble_run(q.copy(), v.copy(), m, dev, [s.planet] * S, [s.asteroid] * S, step_end=5)
    ev, secs = nb.ensemble_run(q, v, m, dev, [s.planet] * S, [s.asteroid] * S, step_end=steps)
    pairs = S * steps * s.n * (s.n - 1)
    print("ensemble %d x %s, %d steps: %.3f s, %.3e pairs/s = %.1f%% of 37.2TF" % (S, case, steps, secs, pairs / secs, pairs / secs * 20 / 37.2e12 * 100), flush=True)


def large(n=65536, steps=10):
    import torch
    n, steps = int(n), int(steps)
    s = nb.synthetic_system(n, seed=42)
    sh = nb.ShardedSystem(s, device="cuda:0")
    sh.advance(3)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    sh.advance(steps)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    pps = n * (n - 1) / (ms * 1e-3)
    print("large n=%d: %.3f ms/step, %.3e pairs/s = %.1f%% of 37.2TF" % (n, ms, pps, pps * 20 / 37.2e12 * 100), flush=True)


def solve(case="b200", gpus=1):
    s = nb.read_input(os.path.join(G, case + ".in"))
    t0 = time.time()
    a = nb.solve(s, gpus=int(gpus))
    print(case, nb.format_output(a.min_dist, a.hit_time_step, a.gravity_device_id, a.missile_cost).replace("\n", " | "),
          "gpu %.3fs wall %.3fs (call %.3fs) %.3e pairs/s" % (a.gpu_seconds, a.wall_seconds, time.time() - t0, a.pair_interactions / a.gpu_seconds), flush=True)


def cli(case="b1024", reps=2):
    """Process wall time of the hw5 binary (CUDA start-up included)."""
    import subprocess
    inp = os.path.join(G, case + ".in")
    for _ in range(int(reps)):
        t0 = time.time()
        r = subprocess.run([nb.HW5_PATH, inp, "/tmp/cli.out"], env=dict(os.environ, NB_VERBOSE="1"), capture_output=True)
        dt = time.time() - t0
        ok = open("/tmp/cli.out").read() == open(os.path.join(G, case + ".out")).read()
        print("hw5 %s: process wall %.3f s, rc %d, byte-identical %s\n%s" % (case, dt, r.returncode, ok, r.stderr.decode().strip()), flush=True)


if __name__ == "__main__":
    globals()[sys.argv[1]](*sys.argv[2:])
