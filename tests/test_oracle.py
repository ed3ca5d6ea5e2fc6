"""CPU: the oracle restatement against the reference-generated goldens, against the star distances and per-sweep
trace recorded in tests/golden/oracle_pins.json and (where oracle/_ref exists) against the reference's own code sweep by
sweep -- which also checks the recorded values."""
import hashlib
import json

import numpy as np
import pytest

import oracle
from uoparallel_seismic_project_b200 import workloads as W

from conftest import ROOT, assert_bit_equal, make_field

PINS = json.loads((ROOT / "tests" / "golden" / "oracle_pins.json").read_text())


def test_restatement_matches_reference_goldens(golden_small):
    for m in golden_small:
        v = make_field(m["kind"], m["dims"], m["seed"])
        assert hashlib.sha256(v.tobytes()).digest() == m["v_sha"], "synthetic field generator drifted"
        tt, sweeps, _ = oracle.solve(v, W.star(m["star"]), m["start"])
        assert_bit_equal(tt, m["tt"], f"{m['case']}[{m['idx']}]")
        assert sweeps == m["ref_sweeps"]


@pytest.mark.skipif(oracle.reference() is None, reason="oracle/_ref not built (needs $SWEEPTT_REFERENCE)")
def test_restatement_sweep_by_sweep_against_reference_code():
    v = W.contrast_field((14, 13, 12), seed=4)
    for name in ("3", "5", "818"):
        off = W.star(name)
        start = (7, 3, 11)
        tt = oracle.init_tt(v.shape, start)
        trace = []
        oracle.ref_solve(v, off, start, per_sweep=lambda k, c, t: trace.append((c, t.copy())))
        for c_ref, t_ref in trace:
            c = oracle.sweep(v, tt, off, start)
            assert c == c_ref
            assert_bit_equal(tt, t_ref, f"{name}-FS per-sweep state")
        assert [[c, hashlib.sha256(t.tobytes()).hexdigest()] for c, t in trace] == PINS["trace"][name]


def test_restatement_sweep_by_sweep_against_recorded_trace():
    case = PINS["trace_case"]
    v = make_field(case["kind"], case["dims"], case["seed"])
    for name in ("3", "5", "818"):
        off = W.star(name)
        tt = oracle.init_tt(v.shape, case["start"])
        for k, (c_ref, sha_ref) in enumerate(PINS["trace"][name]):
            c = oracle.sweep(v, tt, off, case["start"])
            assert c == c_ref, f"{name}-FS sweep {k + 1}: store count"
            assert hashlib.sha256(tt.tobytes()).hexdigest() == sha_ref, f"{name}-FS sweep {k + 1}: field"
        assert c_ref == 0


@pytest.mark.skipif(oracle.reference() is None, reason="oracle/_ref not built")
def test_star_distances_match_reference():
    lib = oracle.reference()
    for name in ("3", "5", "818"):
        off = np.ascontiguousarray(W.star(name), np.int32)
        import ctypes
        assert lib.refh_set_star(ctypes.c_void_p(off.ctypes.data), len(off))
        d_ref = np.array([lib.refh_star_distance(l) for l in range(len(off))], np.float32)
        assert_bit_equal(oracle.star_distances(off), d_ref)
        assert [int(x) for x in d_ref.view(np.uint32)] == PINS["star_distance_bits"][name]


def test_star_distances_match_recorded():
    for name in ("3", "5", "818"):
        want = np.array(PINS["star_distance_bits"][name], np.uint32).view(np.float32)
        assert len(want) == len(W.star(name))
        assert_bit_equal(oracle.star_distances(W.star(name)), want, f"{name}-FS")


def test_fixed_point_invariant_and_detection(golden_small):
    m = golden_small[3]
    v = make_field(m["kind"], m["dims"], m["seed"])
    off = W.star(m["star"])
    assert oracle.violations(v, m["tt"], off, m["start"]) == 0
    worse = m["tt"].copy()
    worse[2, 3, 4] *= 1.5
    assert oracle.violations(v, worse, off, m["start"]) > 0


def test_work_per_sweep_matches_survey():
    # SURVEY.md §3.1 / BASELINE.md: exact visit counts on the 241x241x51 box
    assert oracle.visits_per_sweep((241, 241, 51), W.star("818")) == 2_246_171_812
    assert oracle.visits_per_sweep((241, 241, 51), W.star("3")) == 278_079_410
    assert W.visits_per_sweep((241, 241, 51), W.star("818")) == 2_246_171_812


def test_quirk_missing_edge_is_real():
    """On a constant field, dropping the start-skip/last-offset quirks changes exactly the node
    start - o_last (SURVEY.md §8a.5): the oracle must NOT be 'fixed'."""
    v = W.constant_field((20, 17, 13))
    off = W.star("818")
    start = (12, 9, 11)
    tt, _, _ = oracle.solve(v, off, start)
    n = tuple(np.array(start) - off[-1])
    d = oracle.star_distances(off)
    direct = np.float32(d[-1] * np.float32(0.5)) * np.float32(v[n] + v[start])
    assert tt[n] > direct  # the direct edge {start - o_last, start} is missing from the graph
