"""CPU: the oracle against the reference's goldens (testcases/b*.out) and against the unmodified
reference program (oracle/_ref/nbody = samples/nbody.cc compiled in place) — this is what pins it."""
import json
import os
import subprocess

import numpy as np
import pytest
from conftest import CASES, GOLDEN, case_path, golden_lines


def test_oracle_b20_strict_is_byte_identical_to_golden(oracle, tmp_path):
    """Full 200000-step, three-query run in the reference's exact arithmetic (pow, no FMA)."""
    oracle.lib()
    out = tmp_path / "b20.out"
    subprocess.check_call([oracle.EXE, case_path("b20"), str(out), "200000", "0"])
    assert out.read_text() == golden_lines("b20")["text"]


def test_oracle_b30_sqrt3_mode_is_byte_identical_to_golden(oracle, tmp_path):
    """The sqrt(r2^3) variant (the mode the GPU strict kernel is compared with bit for bit)."""
    oracle.lib()
    out = tmp_path / "b30.out"
    subprocess.check_call([oracle.EXE, case_path("b30"), str(out), "200000", "1"])
    assert out.read_text() == golden_lines("b30")["text"]


def test_committed_kats_cover_all_goldens_byte_identically():
    """tests/golden/oracle_kats.json was produced by make_oracle_kats.py, which aborts unless the
    oracle's three output lines equal testcases/bN.out byte for byte."""
    kats = json.load(open(os.path.join(GOLDEN, "oracle_kats.json")))
    for case in CASES:
        if case not in kats:
            pytest.skip("%s not generated yet" % case)
        k, g = kats[case], golden_lines(case)
        assert k["byte_identical_to_golden"]
        assert float(k["min_dist"]) == g["min_dist"]
        assert k["hit_time_step"] == g["hit_time_step"]
        assert k["gravity_device_id"] == g["gravity_device_id"]
        assert float(k["missile_cost"]) == g["missile_cost"]
        # the golden cost decodes to the reach step of the chosen device (hw5.cu:305)
        if g["gravity_device_id"] >= 0:
            r = [d for d in k["devices"] if d["index"] == g["gravity_device_id"]][0]["reach_step"]
            assert 1e5 + 1e3 * ((r + 1) * 60.0) == g["missile_cost"]


def test_oracle_matches_unmodified_reference_binary_on_b20(oracle, tmp_path):
    """samples/nbody.cc answers queries 1 and 2 only (query 3 is a TODO printing -999).  Its b20 lines are stored in
    golden/reference_b20.json; where the reference tree was present at build time (oracle/_ref/nbody), the program
    itself is run and held to them as well."""
    ref = json.load(open(os.path.join(GOLDEN, "reference_b20.json")))
    g = golden_lines("b20")["text"].split("\n")
    assert ref["lines"] == g[:2]
    assert ref["line3_prefix"] == "-999 "
    oracle.lib()
    out = tmp_path / "oracle.out"
    subprocess.check_call([oracle.EXE, case_path("b20"), str(out), "200000", "0"])
    assert out.read_text().split("\n")[:2] == ref["lines"]
    if os.path.exists(oracle.REF_EXE):
        live = tmp_path / "ref.out"
        subprocess.check_call([oracle.REF_EXE, case_path("b20"), str(live)])
        lines = live.read_text().split("\n")
        assert lines[:2] == ref["lines"] and lines[2].startswith(ref["line3_prefix"])


def test_oracle_step_matches_plain_numpy_restatement(oracle, nb):
    """run_step against an independent numpy transcription of nbody.cc:51-89 on b20 (5 steps)."""
    s = nb.read_input(case_path("b20"))
    q, v = s.q.copy(), s.v.copy()
    oracle.run_steps(oracle.MODE_STRICT, s.n, q, v, s.m, s.is_device, 0, 5, nthreads=1)
    n = s.n
    Q, V = s.q.reshape(3, n).copy(), s.v.reshape(3, n).copy()
    import math
    for step in range(1, 6):
        A = np.zeros((3, n))
        for i in range(n):
            for j in range(n):
                if j == i:
                    continue
                mj = s.m[j]
                if s.is_device[j]:
                    mj = mj + 0.5 * mj * abs(math.sin(step * 60.0 / 6000))
                d = Q[:, j] - Q[:, i]
                dist3 = math.pow(d[0] * d[0] + d[1] * d[1] + d[2] * d[2] + 1e-3 * 1e-3, 1.5)
                for c in range(3):
                    A[c, i] += 6.674e-11 * mj * d[c] / dist3
        V += A * 60.0
        Q += V * 60.0
    assert np.array_equal(Q.reshape(-1), q) and np.array_equal(V.reshape(-1), v)


def test_oracle_modes_agree_bitwise_on_state_b50(oracle, nb):
    """SURVEY App. B: pow(r2,1.5) vs sqrt(r2^3) give the same rounded state on the goldens' magnitudes."""
    s = nb.read_input(case_path("b50"))
    q0, v0 = s.q.copy(), s.v.copy()
    q1, v1 = s.q.copy(), s.v.copy()
    oracle.run_steps(oracle.MODE_STRICT, s.n, q0, v0, s.m, s.is_device, 0, 2000, nthreads=1)
    oracle.run_steps(oracle.MODE_SQRT3, s.n, q1, v1, s.m, s.is_device, 0, 2000, nthreads=1)
    assert np.array_equal(q0, q1)
    # velocities may differ in the last bits (a*dt is far below ulp(q) but not below ulp(v))
    assert np.allclose(v0, v1, rtol=1e-12, atol=0)


def test_oracle_threads_are_bit_identical(oracle, nb):
    s = nb.read_input(case_path("b200"))
    q0, v0 = s.q.copy(), s.v.copy()
    q1, v1 = s.q.copy(), s.v.copy()
    oracle.run_steps(oracle.MODE_STRICT, s.n, q0, v0, s.m, s.is_device, 0, 50, nthreads=1)
    oracle.run_steps(oracle.MODE_STRICT, s.n, q1, v1, s.m, s.is_device, 0, 50, nthreads=4)
    assert np.array_equal(q0, q1) and np.array_equal(v0, v1)


def test_oracle_no_hit_defaults(oracle, nb):
    """hw5.cu:545-548,568: no collision within the horizon -> -2 and '-1 0' (no golden pins this)."""
    s = nb.read_input(case_path("b20"))
    ans = oracle.solve(oracle.MODE_STRICT, s, n_steps=1000)
    assert ans.hit_time_step == -2 and ans.gravity_device_id == -1 and ans.missile_cost == 0.0
