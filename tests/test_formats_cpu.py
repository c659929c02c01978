"""CPU: the generator and the input-format writer (SURVEY.md 8f rank 4).  A generated system written by the
library must be read back bit for bit, and must be a valid input of the UNMODIFIED reference program
(oracle/_ref/nbody) — that is what makes `nbtool gen` files usable on both sides of the drop-in boundary."""
import os
import subprocess

import numpy as np
import pytest
from conftest import GOLDEN


def test_generator_is_deterministic_and_follows_config_c5(nb):
    a, b, c = nb.generate_system(4096, 42), nb.generate_system(4096, 42), nb.generate_system(4096, 43)
    assert np.array_equal(a.q, b.q) and np.array_equal(a.v, b.v) and np.array_equal(a.m, b.m)
    assert not np.array_equal(a.q, c.q)
    assert (a.planet, a.asteroid) == (0, 1)
    assert list(np.nonzero(a.is_device)[0]) == [4092, 4093, 4094, 4095]
    centre = np.array([-2.0e20, -2.9e20, 1.8e18])
    q = a.q.reshape(3, -1)
    assert np.all(np.abs(q - centre[:, None]) <= 0.5e13)
    assert abs(q[0].std() / (1e13 / 12 ** 0.5) - 1) < 0.05           # uniform in the cube
    assert abs(a.v.std() / 1e7 - 1) < 0.03 and abs(a.v.mean()) < 5e5  # N(0, 1e7^2)
    lm = np.log10(a.m)
    assert lm.min() >= 20 and lm.max() <= 30 and abs(lm.mean() - 25) < 0.2  # log-uniform masses
    # known answer: std::mt19937_64(42) raw output is standardised, the transforms are the library's own
    assert a.q[0] == nb.generate_system(2, 42, 0).q[0]


def test_write_input_round_trips_bit_for_bit(nb, tmp_path):
    s = nb.generate_system(300, 7, 3)
    path = tmp_path / "s.in"
    nb.write_input(str(path), s)
    t = nb.read_input(str(path))
    assert (t.n, t.planet, t.asteroid) == (s.n, s.planet, s.asteroid)
    for x, y in ((s.q, t.q), (s.v, t.v), (s.m, t.m), (s.is_device, t.is_device)):
        assert np.array_equal(x, y)
    head = path.read_text().split("\n")
    assert head[0] == "300 0 1" and head[1].endswith(" planet") and head[2].endswith(" asteroid") and head[300].endswith(" device")


def test_nbtool_gen_writes_the_same_file_as_the_library(nb, tmp_path):
    a, b = tmp_path / "a.in", tmp_path / "b.in"
    subprocess.check_call([nb.NBTOOL_PATH, "gen", "64", "9", str(a), "2"])
    nb.write_input(str(b), nb.generate_system(64, 9, 2))
    assert a.read_bytes() == b.read_bytes()
    assert subprocess.run([nb.NBTOOL_PATH, "frobnicate"], capture_output=True).returncode == 2


def test_nbtool_gen_writes_the_stored_vector(nb, tmp_path):
    """The file the test below feeds to the reference program is pinned byte for byte (generator and writer)."""
    out = tmp_path / "g.in"
    subprocess.check_call([nb.NBTOOL_PATH, "gen", "5", "3", str(out), "1"])
    assert out.read_bytes() == open(os.path.join(GOLDEN, "gen_5_3_1.in"), "rb").read()


def test_generated_file_is_a_valid_input_of_the_unmodified_reference(nb, oracle, tmp_path):
    """samples/nbody.cc (compiled in place as oracle/_ref/nbody) and the oracle restatement read the generated file
    and agree on output lines 1-2 (the sample leaves query 3 as a TODO)."""
    if not os.path.exists(oracle.REF_EXE):
        pytest.skip("oracle/_ref/nbody not built (reference tree absent)")
    oracle.lib()
    inp, ref_out, ora_out = tmp_path / "g.in", tmp_path / "ref.out", tmp_path / "ora.out"
    subprocess.check_call([nb.NBTOOL_PATH, "gen", "5", "3", str(inp), "1"])
    subprocess.check_call([oracle.REF_EXE, str(inp), str(ref_out)], timeout=120)
    subprocess.check_call([oracle.EXE, str(inp), str(ora_out), "200000", "0"], timeout=120)
    assert ref_out.read_text().split("\n")[:2] == ora_out.read_text().split("\n")[:2]
