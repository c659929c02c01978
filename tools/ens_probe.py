"""Ensemble of 1024-body systems on one GPU (the symmetric single-block kernel)."""
import importlib, os, sys, time
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
nb = importlib.import_module("nthu_ipc_nbody-simulation_b200")
S = int(sys.argv[1]) if len(sys.argv) > 1 else 148
steps = int(sys.argv[2]) if len(sys.argv) > 2 else 1000
base = nb.read_input(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "testcases", "b1024.in"))
q = np.tile(base.q, (S, 1)); v = np.stack([base.v * (1 + 1e-9 * k) for k in range(S)])
m = np.tile(base.m, (S, 1)); dev = np.tile(base.is_device, (S, 1))
nb.ensemble_run(q.copy(), v.copy(), m, dev, [base.planet] * S, [base.asteroid] * S, kind=nb.KIND_Q2, step_end=20)
ev, secs = nb.ensemble_run(q, v, m, dev, [base.planet] * S, [base.asteroid] * S, kind=nb.KIND_Q2, step_end=steps)
pairs = S * steps * 1024 * 1023
print("%d systems x %d steps: %.3f s, %.1f us/step, %.3e pairs/s = %.1f%% of 37.2 TF" % (
    S, steps, secs, secs / steps * 1e6 / max(1, -(-S // 148)), pairs / secs, pairs / secs * 20 / 37.2e12 * 100))
