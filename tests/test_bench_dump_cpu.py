"""CPU: bench.py --dump-outputs writes the planar state as float64 [3, n] arrays, sampled the same way for q and v
above the size limit."""
import numpy as np

import bench


def test_dump_state_writes_the_planar_state(tmp_path):
    n = 1000
    q = np.arange(3 * n, dtype=np.float64)
    bench.dump_state(np, str(tmp_path), q, -q, n)
    a, b = np.load(tmp_path / "positions.npy"), np.load(tmp_path / "velocities.npy")
    assert a.dtype == b.dtype == np.float64 and a.shape == b.shape == (3, n)
    assert np.array_equal(a, q.reshape(3, n)) and np.array_equal(b, -a)


def test_dump_state_samples_the_same_bodies_above_the_limit(tmp_path, monkeypatch):
    n, keep = 1000, 100
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", keep * 2 * 3 * 8)
    q = np.arange(3 * n, dtype=np.float64)
    bench.dump_state(np, str(tmp_path / "a"), q, -q, n)
    bench.dump_state(np, str(tmp_path / "b"), q, -q, n)
    a, b = np.load(tmp_path / "a" / "positions.npy"), np.load(tmp_path / "a" / "velocities.npy")
    assert a.shape == b.shape == (3, keep) and a.nbytes + b.nbytes <= bench.DUMP_LIMIT_BYTES
    idx = a[0].astype(np.int64)  # body index, since q[0, i] == i
    assert np.all(np.diff(idx) > 0) and np.array_equal(a, q.reshape(3, n)[:, idx]) and np.array_equal(b, -a)
    assert np.array_equal(a, np.load(tmp_path / "b" / "positions.npy"))  # the sample is fixed
