"""CPU: file formats of the drop-in surface (csrc/hostio.cpp through the C ABI) against the
oracle's restatement, the .vbox bytes recorded in tests/golden/oracle_pins.json and -- where oracle/_ref exists -- the
reference's own loaders/writers."""
import ctypes
import hashlib
import json
import struct
import subprocess

import numpy as np
import pytest

import oracle
import uoparallel_seismic_project_b200 as P
from uoparallel_seismic_project_b200 import workloads as W

from conftest import ROOT

VBOX_SHA = json.loads((ROOT / "tests" / "golden" / "oracle_pins.json").read_text())["vbox_sha256"]


def _sha(path):
    return hashlib.sha256(path.read_bytes()).hexdigest()


def test_vbox_store_bytes_match_oracle_and_vconvert(tmp_path):
    v = (W.random_field((7, 5, 9), seed=3) - np.float32(0.25)).astype(np.float32)  # negative values: sign-extension matters
    P.vbox_store(tmp_path / "ours.vbox", v, origin=(1, 1, 1))
    oracle.vbox_write(tmp_path / "oracle.vbox", v, origin=(1, 1, 1))
    assert (tmp_path / "ours.vbox").read_bytes() == (tmp_path / "oracle.vbox").read_bytes()
    assert _sha(tmp_path / "ours.vbox") == VBOX_SHA["vbox_store_random_7x5x9_seed3_minus_quarter"]
    vc = oracle.vconvert_path()
    if vc is not None:  # the reference's own tools/vconvert.c on the same text input
        W.write_text_a(tmp_path / "v.txt", v)
        subprocess.run([str(vc), str(tmp_path / "v.txt"), str(tmp_path / "ref.vbox")], check=True, capture_output=True)
        assert (tmp_path / "ref.vbox").read_bytes() == (tmp_path / "ours.vbox").read_bytes()


def test_vconvert_tool_matches_reference_tool(tmp_path):
    v = W.heterogeneous_field((5, 6, 7), seed=9)
    W.write_text_a(tmp_path / "v.txt", v)
    ours = P.lib_path().parent / "vconvert"
    r = subprocess.run([str(ours), str(tmp_path / "v.txt"), str(tmp_path / "ours.vbox")], capture_output=True, text=True)
    assert r.returncode == 0 and "writing new velocity model" in r.stdout
    got, origin, dims = P.vbox_load(tmp_path / "ours.vbox")
    assert origin == (1, 1, 1) and np.array_equal(got, v)
    assert _sha(tmp_path / "ours.vbox") == VBOX_SHA["vconvert_hetero_5x6x7_seed9"]
    vc = oracle.vconvert_path()
    if vc is not None:
        subprocess.run([str(vc), str(tmp_path / "v.txt"), str(tmp_path / "ref.vbox")], check=True, capture_output=True)
        assert (tmp_path / "ref.vbox").read_bytes() == (tmp_path / "ours.vbox").read_bytes()


def test_vbox_checksum_is_the_sign_extended_sum(tmp_path):
    v = np.array([[[-1.5, 2.0, -3.25]]], np.float32)
    P.vbox_store(tmp_path / "a.vbox", v)
    raw = (tmp_path / "a.vbox").read_bytes()
    words = raw[:-4]
    s = 0
    for i in range(0, len(words), 4):
        b = struct.unpack("4b", words[i:i + 4])  # signed bytes, include/velocityboxfiler.h:78-83,248-251
        s = (s + b[0] + (b[1] << 8) + (b[2] << 16) + (b[3] << 24)) & 0xFFFFFFFF
    assert struct.unpack("<I", raw[-4:])[0] == s
    plain = sum(struct.unpack(f"<{len(words)//4}I", words)) & 0xFFFFFFFF
    assert plain != s  # not a plain uint32 sum


def test_vbox_load_roundtrip_and_rejects(tmp_path):
    v = W.heterogeneous_field((6, 7, 8), seed=2)
    P.vbox_store(tmp_path / "a.vbox", v, origin=(1, 2, 3))
    got, origin, dims = P.vbox_load(tmp_path / "a.vbox")
    assert origin == (1, 2, 3) and dims == (6, 7, 8) and np.array_equal(got, v)
    assert oracle.vbox_read(tmp_path / "a.vbox")[0].tobytes() == v.tobytes()
    raw = bytearray((tmp_path / "a.vbox").read_bytes())
    raw[40] ^= 0x10
    (tmp_path / "bad.vbox").write_bytes(raw)
    with pytest.raises(P.SweepError, match="checksum"):
        P.vbox_load(tmp_path / "bad.vbox")
    (tmp_path / "magic.vbox").write_bytes(b"xbov" + bytes(raw[4:]))
    with pytest.raises(P.SweepError, match="not a vbox"):
        P.vbox_load(tmp_path / "magic.vbox")
    (tmp_path / "short.vbox").write_bytes(bytes(raw[:-20]))
    with pytest.raises(P.SweepError):
        P.vbox_load(tmp_path / "short.vbox")
    with pytest.raises(P.SweepError, match="opening"):
        P.vbox_load(tmp_path / "missing.vbox")


@pytest.mark.skipif(oracle.reference() is None, reason="oracle/_ref not built")
def test_reference_loader_accepts_our_vbox(tmp_path):
    v = W.random_field((5, 4, 6), seed=8)
    P.vbox_store(tmp_path / "a.vbox", v, origin=(1, 1, 1))
    lib = oracle.reference()
    dims, origin = (ctypes.c_int * 3)(), (ctypes.c_int * 3)()
    assert lib.refh_load_vbox(str(tmp_path / "a.vbox").encode(), dims, origin)
    assert tuple(dims) == (5, 4, 6) and tuple(origin) == (1, 1, 1)
    got = np.ctypeslib.as_array(lib.refh_velocity_ptr(), shape=(v.size,)).reshape(v.shape)
    assert np.array_equal(got, v)
    assert _sha(tmp_path / "a.vbox") == VBOX_SHA["vbox_store_random_5x4x6_seed8"]


def test_vbox_bytes_match_the_recorded_file_the_reference_loader_reads(tmp_path):
    """The file test_reference_loader_accepts_our_vbox hands to the reference's loader, against the recorded bytes."""
    P.vbox_store(tmp_path / "a.vbox", W.random_field((5, 4, 6), seed=8), origin=(1, 1, 1))
    assert _sha(tmp_path / "a.vbox") == VBOX_SHA["vbox_store_random_5x4x6_seed8"]


def test_vbox_subset(tmp_path):
    v = W.random_field((9, 8, 7), seed=4)
    P.vbox_store(tmp_path / "a.vbox", v)
    sub = P.vbox_load_subset(tmp_path / "a.vbox", (3, 2, 1), (3, 4, 5))  # "middle third" like examples/example_velocityboxfiler.c
    assert np.array_equal(sub, v[3:6, 2:6, 1:6])
    with pytest.raises(P.SweepError, match="subset"):
        P.vbox_load_subset(tmp_path / "a.vbox", (7, 0, 0), (3, 1, 1))


def test_text_dialects(tmp_path):
    v = W.random_field((4, 3, 5), seed=6)
    W.write_text_a(tmp_path / "a.txt", v)
    got, origin, dims = P.text_load(tmp_path / "a.txt")
    assert origin == (1, 1, 1) and dims == (4, 3, 5) and np.array_equal(got, v)
    W.write_text_b(tmp_path / "b.txt", v)
    got, origin, dims = P.text_load(tmp_path / "b.txt")
    assert origin == (0, 0, 0) and dims == (4, 3, 5) and np.array_equal(got, v)
    ref = oracle.reference()
    if ref is not None:
        d, o = (ctypes.c_int * 3)(), (ctypes.c_int * 3)()
        assert ref.refh_load_text(str(tmp_path / "a.txt").encode(), d, o)
        r = np.ctypeslib.as_array(ref.refh_velocity_ptr(), shape=(v.size,)).reshape(v.shape)
        assert np.array_equal(r, got) and tuple(d) == (4, 3, 5) and tuple(o) == (1, 1, 1)
    (tmp_path / "c.txt").write_text("1,1,1,0.5\n1,1,2,oops\n")
    with pytest.raises(P.SweepError, match="confused by line 2"):
        P.text_load(tmp_path / "c.txt")


def test_star_and_start_files(tmp_path):
    for name in ("3", "5", "818"):
        W.write_star_file(tmp_path / "fs.txt", W.star(name))
        off, d = P.star_load(tmp_path / "fs.txt")
        assert np.array_equal(off, W.star(name))
        assert d.tobytes() == oracle.star_distances(W.star(name)).tobytes()
    W.write_start_file(tmp_path / "st.txt", W.starts(111))
    assert np.array_equal(P.starts_load(tmp_path / "st.txt"), W.starts(111))
    with pytest.raises(P.SweepError, match="Cannot open forward star offset file"):
        P.star_load(tmp_path / "nope.txt")
    (tmp_path / "trunc.txt").write_text("5\n1 0 0\n0 1 0\n")
    with pytest.raises(P.SweepError):
        P.starts_load(tmp_path / "trunc.txt")


def test_output_tt_bytes_match_reference_format(tmp_path):
    rng = np.random.default_rng(1)
    tt = (rng.random((2, 5, 4, 6)) * 3000).astype(np.float32)
    tt[0, 0, 0, 0] = 0.0
    tt[1, 1, 1, 1] = np.inf
    tt[1, 2, 2, 2] = np.float32(1e-7)
    tt[0, 4, 3, 5] = np.float32(123456.789)
    P.write_output_tt(tmp_path / "ours.tt", tt)
    oracle.write_output_tt(tmp_path / "oracle.tt", tt)
    assert (tmp_path / "ours.tt").read_bytes() == (tmp_path / "oracle.tt").read_bytes()
    first = (tmp_path / "ours.tt").read_text().splitlines()[:3]
    assert first == ["5 4 6", "starting point: 0", "travel time for (0,0,0): 0.000000 0 0 0"]


def test_fast_float_formatter_is_printf_exact(tmp_path):
    """The writer formats %f with exact integer arithmetic; compare with printf on hard cases."""
    rng = np.random.default_rng(7)
    bits = rng.integers(0, 0x7F800000, size=40000, dtype=np.uint32)
    vals = np.concatenate([bits.view(np.float32), -bits[:2000].view(np.float32),
                           np.array([0.0, -0.0, 0.5e-6, 1.5e-6, 2.5e-6, 0.0000005, 0.1, 1e10, 3e38, 2**39, 2**40 - 1,
                                     np.inf, -np.inf, 0.125, 0.0000015, 8388608.5, 1234.5678], np.float32)])
    vals = vals.reshape(1, 1, 1, -1)
    P.write_output_tt(tmp_path / "a.tt", vals)
    lines = (tmp_path / "a.tt").read_text().splitlines()[2:]
    for x, line in zip(vals.ravel(), lines):
        assert line.split(": ")[1].split(" ")[0] == "%f" % float(x), (x, line)
