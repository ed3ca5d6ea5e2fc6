"""The ray, tomography, ray-set and location operators at the float edges and size boundaries of their contracts
(include/sweeptt.h; DESIGN §3.8-3.10).

The yardsticks are the CPU oracles of the other suites (oracle_rays, oracle_project, oracle_backproject, quantum_exp,
round_once, oracle_misfit / oracle_locate) and exact rational arithmetic where a claim is about rounding; every
comparison is bit for bit, except that a NaN projection equals a NaN oracle value whatever the payloads.
CPU: round_once against exact rational rounding over the subnormal and overflow ranges; loc_div / loc_remainder
restated operation for operation in numpy float64 against correctly rounded a / k on over 10^6 pairs, the hardest
ones (quotients nearest a midpoint, just below a power of two) included.
GPU (-m gpu): rays longer than one 32-edge walk round (a straight line with every length 1..200, a long thin box, the
maze) under both kernels, with max_nodes on both sides of 31..65-node rays; back-projection of subnormal, huge,
overflowing and cancelling weights and at delta = 1e-20 / 1e20, and single rays whose node value lands exactly on a
rounding boundary; projection of signed zeros, infinities, NaN, subnormals and overflowing sums; ray sets frozen in
many chunks (prime size, chunks with no OK ray, one ray per chunk); location at every kernel-shape switch and at the
station limit, with overflowing, subnormal and signed-zero misfits and origin times against numpy's a / k for every
k up to the limit; put_tt refusing NaN and negative times and leaving the context as it was.  The GPU tests take 10 s
on one B200 (1000 W power limit)."""
import math
from fractions import Fraction

import numpy as np
import pytest

import oracle
import uoparallel_seismic_project_b200 as P
from uoparallel_seismic_project_b200 import api, workloads as W

from conftest import make_field
from test_locate import _bits32, _fields, assert_locations_equal, oracle_locate, oracle_misfit
from test_rays import _golden_cases, all_nodes, oracle_rays
from test_tomography import (AXIS_STAR, _bits_equal, _ctx, _hd_max, _maze, _weights, oracle_backproject,
                             oracle_project, quantum_exp, round_once)

gpu = pytest.mark.gpu
OK, UNREACHED, TRUNCATED = api.RAY_OK, api.RAY_UNREACHED, api.RAY_TRUNCATED
F = np.float32
FMAX = float(np.finfo(np.float32).max)
TINY = 2.0 ** -149
LOC_MAX_STATIONS = 904   # include/sweeptt.h: the largest station count sweeptt_locate_events accepts on a B200
STAGING = 1 << 28        # the library's freeze staging, bytes: a chunk is max(1, STAGING / (2 max_nodes)) rays


# ---- exact references --------------------------------------------------------------------------

def exact_float32(x: Fraction) -> np.float32:
    """The float32 nearest to the rational x (ties to even; +-INF from FLT_MAX + half an ulp on), without any
    floating-point rounding of x itself."""
    if x == 0:
        return np.float32(0.0)
    a = abs(x)
    e = a.numerator.bit_length() - a.denominator.bit_length()
    while Fraction(2) ** e > a:
        e -= 1
    while Fraction(2) ** (e + 1) <= a:
        e += 1
    q = Fraction(2) ** max(e - 23, -149)   # quantum of a's binade, or of the subnormals
    n = a / q
    r = n.numerator // n.denominator
    rem = n - r
    if rem > Fraction(1, 2) or (rem == Fraction(1, 2) and r % 2):
        r += 1
    mag = r * q
    out = np.float32(np.inf) if mag >= Fraction(2) ** 128 else np.float32(math.ldexp(r, int(math.log2(q))))
    assert out == np.inf or Fraction(float(out)) == mag
    return -out if x < 0 else out


def np_loc_remainder(a, q, k):
    """kernels.cu loc_remainder, in numpy float64 (no contraction): a - q*k exactly, q split by Veltkamp."""
    c = 134217729.0 * q
    qh = c - (c - q)
    ql = q - qh
    return (a - qh * k) - ql * k


def np_loc_div(a, k):
    """kernels.cu loc_div, operation for operation: q = a * RN(1/k), then at most four steps to the neighbour towards
    a / k while it is nearer (elementwise over arrays a, k; k >= 1)."""
    a = np.asarray(a, np.float64)
    kd = np.asarray(k, np.float64)
    q = a * (1.0 / kd)
    r = np_loc_remainder(a, q, kd)
    live = r != 0.0
    for _ in range(4):
        step = np.where((r > 0.0) == (q > 0.0), 1, -1).astype(np.int64)
        qn = (q.view(np.int64) + step).view(np.float64)
        rn = np_loc_remainder(a, qn, kd)
        take = live & (np.abs(rn) < np.abs(r))
        q = np.where(take, qn, q)
        r = np.where(take, rn, r)
        live = take & (r != 0.0)
    return q


def _hard_dividends(k, rng, n):
    """Dividends a (doubles) whose quotient a/k lies nearest a midpoint between two doubles, and just below a power
    of two: for each of n binades the best of a = RN(k * M) and its 6 neighbours, by exact rational distance."""
    out = []
    for _ in range(n):
        p = int(rng.integers(-140, 120))
        mid = Fraction(2 * int(rng.integers(1 << 52, 1 << 53)) + 1) * Fraction(2) ** (p - 53)   # (2i+1) 2^(p-53)
        a0 = float(mid * k)
        best, bd = a0, None
        for j in range(-3, 4):
            a = float((np.array([a0]).view(np.int64) + j).view(np.float64)[0])
            qx = Fraction(a) / k
            ulp = Fraction(2) ** (math.frexp(float(qx))[1] - 53)
            dist = abs(qx / ulp - (qx / ulp).__floor__() - Fraction(1, 2))
            if bd is None or dist < bd:
                best, bd = a, dist
        out.append(best)
        below = float(Fraction(2) ** p * k)   # a/k just below 2^p: the first dividends under k 2^p
        for j in (1, 2, 3):
            out.append((np.array([below]).view(np.int64) - j).view(np.float64)[0])
    return out


# ---- CPU ---------------------------------------------------------------------------------------

def test_round_once_is_exact_rational_rounding_in_the_subnormals_and_at_overflow():
    rng = np.random.default_rng(21)
    cases = []
    for _ in range(3000):   # |total * 2^e| from 2^-160 to 2^-120: subnormals and the smallest normals
        bits = int(rng.integers(1, 63))
        total = int(rng.integers(1 << (bits - 1), 1 << bits)) * int(rng.choice([-1, 1]))
        cases.append((total, int(rng.integers(-160, -119)) - bits))
    for _ in range(3000):   # around FLT_MAX and 2^128
        bits = int(rng.integers(24, 63))
        total = int(rng.integers(1 << (bits - 1), 1 << bits)) * int(rng.choice([-1, 1]))
        cases.append((total, 127 - bits + int(rng.integers(0, 3))))
    # the boundaries themselves: half a subnormal quantum, 1.5 quanta, just below 2^-126 (ties up to the smallest
    # normal), FLT_MAX + half an ulp (ties to even: INF) and just below it
    for t in (1, 3, 5, (1 << 24) - 1, (1 << 24) - 3, (1 << 48) - 1):
        cases += [(t, -150), (t, -150 - (t.bit_length() - 1) // 24 * 24)]
    cases += [((1 << 25) - 1, 103), ((1 << 25) - 2, 103), ((1 << 26) - 1, 102), (((1 << 25) - 1) << 30, 73),
              ((((1 << 25) - 1) << 30) - 1, 73), (1, 128), (-1, 128), (-((1 << 25) - 1), 103)]
    n_sub = n_inf = 0
    for total, e in cases:
        want = exact_float32(Fraction(total) * Fraction(2) ** e)
        got = round_once(total, e)
        assert got.view(np.uint32) == want.view(np.uint32), (total, e, got, want)
        n_sub += bool(0 < abs(float(want)) < 2.0 ** -126)
        n_inf += bool(np.isinf(want))
    assert n_sub > 1000 and n_inf > 500
    assert round_once((1 << 25) - 1, 103) == np.inf and round_once((1 << 25) - 2, 103) == np.float32(FMAX)


def test_exact_float32_agrees_with_numpy_where_a_double_holds_the_value():
    rng = np.random.default_rng(22)
    for _ in range(2000):
        x = float(rng.uniform(0.5, 1)) * 2.0 ** int(rng.integers(-160, 130)) * float(rng.choice([-1, 1]))
        with np.errstate(over="ignore"):
            want = np.float32(x)   # one rounding of an exact double
        assert exact_float32(Fraction(x)).view(np.uint32) == want.view(np.uint32), x


def test_loc_div_restated_is_correctly_rounded_on_a_million_pairs():
    """a / k for k over 1..904 and up to 2^26 - 1, |a| from 2^-149 to 904 * 2^129, both signs."""
    rng = np.random.default_rng(23)
    n = 1 << 20
    k = np.concatenate([np.arange(1, 905), rng.integers(1, 905, n // 2 - 904), rng.integers(905, 1 << 26, n // 2)])
    mant = rng.uniform(1.0, 2.0, n)
    a = mant * np.exp2(rng.integers(-149, 140, n).astype(np.float64)) * rng.choice([-1.0, 1.0], n)
    a[:1000] = rng.integers(-(1 << 40), 1 << 40, 1000).astype(np.float64) * k[:1000]   # exact multiples: r = 0
    got = np_loc_div(a, k)
    want = a / k.astype(np.float64)
    bad = np.nonzero(got.view(np.int64) != want.view(np.int64))[0]
    assert len(bad) == 0, [(a[i], k[i], got[i], want[i]) for i in bad[:5]]


def test_loc_div_restated_on_the_hardest_quotients():
    rng = np.random.default_rng(24)
    ks = list(range(1, 905)) + [int(x) for x in rng.integers(905, 1 << 26, 60)] + [(1 << 26) - 1, 3 * 5 * 7 * 11 * 13]
    a_all, k_all = [], []
    for k in ks:
        for a in _hard_dividends(k, rng, 2):
            a_all.append(a)
            k_all.append(k)
    a_all, k_all = np.array(a_all), np.array(k_all)
    got = np_loc_div(a_all, k_all)
    want = a_all / k_all.astype(np.float64)
    assert (got.view(np.int64) == want.view(np.int64)).all()
    for i in rng.choice(len(a_all), 300, replace=False):   # numpy's quotient is the correctly rounded one
        qx = Fraction(float(a_all[i])) / int(k_all[i])
        lo, hi = np.nextafter(want[i], -np.inf), np.nextafter(want[i], np.inf)
        assert abs(Fraction(float(want[i])) - qx) <= min(abs(Fraction(float(lo)) - qx), abs(Fraction(float(hi)) - qx))


# ---- GPU helpers -------------------------------------------------------------------------------

def _line(n, seed=0, delta=10.0):
    """An (n, 1, 1) box with the six axis offsets: every ray is the straight line to x = 0, so the receivers at every
    x give every length 1..n."""
    v = np.random.default_rng(seed).uniform(0.2, 0.4, (n, 1, 1)).astype(F)
    rec = np.array([(x, 0, 0) for x in range(n)], np.int32)
    return v, AXIS_STAR, (0, 0, 0), rec, delta


def _thin():
    """A 300 x 3 x 3 box with the 3-FS star: long diagonal paths."""
    v = make_field("random", (300, 3, 3), 31)
    return v, W.star("3"), (0, 1, 1), all_nodes(v.shape), 10.0


def _maze_case():
    v = _maze()
    return v, AXIS_STAR, (0, 0, 0), all_nodes(v.shape), 10.0


def _context(v, star, starts, delta=10.0, kernel=None):
    ctx = P.SweepContext(kernel=kernel)
    ctx.set_model(v); ctx.set_star(star, delta); ctx.set_sources(starts)
    ctx.run()
    return ctx


def _nan_or_bits_equal(a, b):
    a, b = np.asarray(a, F), np.asarray(b, F)
    both = np.isnan(a) & np.isnan(b)
    return bool(((a.view(np.uint32) == b.view(np.uint32)) | both).all())


def _assert_set_equals(rs, tr, pd, bp, d, w, what):
    """A frozen set against trace_rays / ray_project / ray_backproject of the same receivers and max_nodes."""
    assert (rs.status == tr.status).all() and (rs.length == tr.length).all() and _bits_equal(rs.tt, tr.tt), what
    offsets, nodes = rs.paths()
    ok = (rs.status == OK).ravel()
    flat = tr.nodes.reshape(-1, tr.nodes.shape[2], 3)
    want = [flat[q, :rs.length.ravel()[q]] for q in np.nonzero(ok)[0]]
    assert (nodes == np.concatenate(want or [np.zeros((0, 3), np.int32)])).all(), f"{what}: paths"
    assert _bits_equal(rs.project(d).values, pd.values), f"{what}: set projection"
    sb = rs.backproject(w)
    assert sb.quantum_exp == bp.quantum_exp and _bits_equal(sb.grad, bp.grad), f"{what}: set back-projection"


def _check_against_oracle(ctx, v, star, start, rec, delta, max_nodes, seed, what):
    """trace_rays, a signed projection and a mixed back-projection against the oracle, then a frozen set."""
    tt = ctx.get_tt(0)
    nodes, length, status, ttr = oracle_rays(v, tt, star, start, rec, delta=delta, max_nodes=max_nodes)
    tr = ctx.trace_rays(rec, max_nodes=max_nodes)
    assert (tr.status[0] == status).all() and (tr.length[0] == length).all(), what
    assert (tr.nodes[0] == nodes).all() and _bits_equal(tr.tt[0], ttr), f"{what}: nodes"
    rng = np.random.default_rng(seed)
    d = (rng.standard_normal(v.shape) * 2.0 ** rng.integers(-8, 9, v.shape)).astype(F)
    w = _weights((1, len(rec)), seed + 1)
    pd = ctx.ray_project(d, rec, max_nodes=max_nodes)
    assert _nan_or_bits_equal(pd.values[0], oracle_project(d, nodes, length, status, delta)), f"{what}: projection"
    bp = ctx.ray_backproject(w, rec, max_nodes=max_nodes)
    g, e = oracle_backproject(v.shape, [(nodes, length, status)], w, _hd_max(star, delta), delta)
    assert bp.quantum_exp == e and _bits_equal(bp.grad, g), f"{what}: back-projection"
    with ctx.freeze_rays(rec, max_nodes=max_nodes) as rs:
        _assert_set_equals(rs, tr, pd, bp, d, w, what)
    return length, status


# ---- GPU: rays longer than one walk round ------------------------------------------------------

@gpu
@pytest.mark.parametrize("kernel", [api.KERNEL_SIMPLE, api.KERNEL_TILED])
@pytest.mark.parametrize("case", ["line", "thin", "maze"])
def test_rays_of_many_rounds_equal_the_oracle(case, kernel):
    v, star, start, rec, delta = {"line": lambda: _line(200, 1), "thin": _thin, "maze": _maze_case}[case]()
    cap = 4 * sum(v.shape)
    with _context(v, star, [start], delta, kernel) as ctx:
        length, status = _check_against_oracle(ctx, v, star, start, rec, delta, cap, 40, f"{case} kernel={kernel}")
    assert (status == OK).any() and length[status == OK].max() > 32, (case, length.max())
    if case == "line":
        assert sorted(length) == list(range(1, 201))


@gpu
def test_max_nodes_on_both_sides_of_the_walk_rounds():
    v, star, start, rec, delta = _line(70, 2)
    with _context(v, star, [start], delta) as ctx:
        for L in (31, 32, 33, 64, 65):
            for cap in (L - 1, L, L + 1):
                what = f"L={L} max_nodes={cap}"
                length, status = _check_against_oracle(ctx, v, star, start, rec, delta, cap, L + cap, what)
                assert status[L - 1] == (OK if cap >= L else TRUNCATED) and length[L - 1] == min(L, cap), what


# ---- GPU: back-projection at the extremes ------------------------------------------------------

def _extreme_weights(R, rng):
    sign = rng.choice(np.array([-1, 1], F), R)
    half = R // 2
    cancel = np.concatenate([rng.standard_normal(half), np.zeros(R - half)]).astype(F)
    cancel[half:2 * half] = -cancel[:half]   # with the receivers listed twice: every contribution cancels
    return {"all 2^-149": np.full(R, TINY, F),
            "FLT_MAX and 2^-149": np.where(rng.random(R) < 0.5, F(FMAX), F(TINY)).astype(F),
            "+-FLT_MAX": (sign * F(FMAX)).astype(F),
            "cancelling": cancel}


@gpu
@pytest.mark.parametrize("delta", [10.0, 1e-20, 1e20])
def test_back_projection_of_extreme_weights_equals_the_oracle(delta):
    v, star, start, rec1, _ = _line(80, 3)
    rec = np.concatenate([rec1, rec1])   # every ray twice: the cancelling weights meet at every node
    R = len(rec)
    hd_max = _hd_max(star, delta)
    with _context(v, star, [start], delta) as ctx:
        tt = ctx.get_tt(0)
        nodes, length, status, _ = oracle_rays(v, tt, star, start, rec, delta=delta)
        assert (status == OK).all()
        with ctx.freeze_rays(rec) as rs:
            for name, w in _extreme_weights(R, np.random.default_rng(5)).items():
                w = w[None, :]
                g, e = oracle_backproject(v.shape, [(nodes, length, status)], w, hd_max, delta)
                assert e == quantum_exp(hd_max, float(np.abs(w).max()), R)
                bp, sb = ctx.ray_backproject(w, rec), rs.backproject(w)
                what = f"{name} delta={delta}"
                assert bp.quantum_exp == e and _bits_equal(bp.grad, g), f"{what}: operator"
                assert sb.quantum_exp == e and _bits_equal(sb.grad, g), f"{what}: ray set"
                if name == "cancelling":
                    assert (g.view(np.uint32) == 0).all(), "exact cancellation is +0, never -0"
                if name == "+-FLT_MAX" and delta == 10.0:
                    assert np.isinf(g).any()
            w = _weights((1, R), 6)   # the mixed weights of the other suites, at this delta
            g, e = oracle_backproject(v.shape, [(nodes, length, status)], w, hd_max, delta)
            bp = ctx.ray_backproject(w, rec)
            assert bp.quantum_exp == e and _bits_equal(bp.grad, g) and _bits_equal(rs.backproject(w).grad, g)


@gpu
def test_single_rays_land_on_the_rounding_boundaries():
    """delta = 1, so an axis edge has hd = 1/2 and a node's value is an exact sum of w/2 terms.  Receivers x = 1, 2 on a
    line from x = 0: node 1 gets w_1/2 (receiver end) + w_2 (two interior edges)."""
    v, star, start, _, _ = _line(4, 4, 1.0)
    rec = np.array([(1, 0, 0), (2, 0, 0)], np.int32)
    cases = {  # (w_1, w_2) -> what node 1 must round to
        "half a subnormal quantum": ((TINY, 0.0), 0.0),
        "1.5 quanta": ((3 * TINY, 0.0), 2 * TINY),
        "just below 2^-126": (((2 ** 24 - 1) * TINY, 0.0), 2.0 ** -126),
        "1.5 quanta below 2^-126": (((2 ** 24 - 3) * TINY, 0.0), (2 ** 23 - 2) * TINY),
        "FLT_MAX + half an ulp": ((2.0 ** 104, FMAX), np.inf),
        "below FLT_MAX + half an ulp": ((2.0 ** 104 * (1 - 2.0 ** -24), FMAX), FMAX),
        "-FLT_MAX - half an ulp": ((-2.0 ** 104, -FMAX), -np.inf),
    }
    with _context(v, star, [start], 1.0) as ctx:
        nodes, length, status, _ = oracle_rays(v, ctx.get_tt(0), star, start, rec, delta=1.0)
        with ctx.freeze_rays(rec) as rs:
            for name, ((w1, w2), want) in cases.items():
                w = np.array([[w1, w2]], F)
                assert float(w[0, 0]) == w1 and float(w[0, 1]) == w2, name
                g, e = oracle_backproject(v.shape, [(nodes, length, status)], w, 0.5, 1.0)
                assert g[1, 0, 0].view(np.uint32) == np.float32(want).view(np.uint32), (name, g[1, 0, 0])
                bp, sb = ctx.ray_backproject(w, rec), rs.backproject(w)
                assert bp.quantum_exp == e and _bits_equal(bp.grad, g), f"{name}: operator {bp.grad.ravel()}"
                assert sb.quantum_exp == e and _bits_equal(sb.grad, g), f"{name}: ray set"


# ---- GPU: projection of special values ---------------------------------------------------------

def _special_perturbations(n, rng):
    base = rng.standard_normal((n, 1, 1)).astype(F)
    out = {"+0": np.zeros((n, 1, 1), F), "-0": np.full((n, 1, 1), -0.0, F),
           "+-0": rng.choice(np.array([0.0, -0.0], F), (n, 1, 1)),
           "2^-149": np.full((n, 1, 1), TINY, F), "FLT_MAX": np.full((n, 1, 1), FMAX, F)}
    for name, at in (("+INF", {7: np.inf}), ("-INF", {40: -np.inf}), ("+INF,-INF", {7: np.inf, 40: -np.inf}),
                     ("NaN", {20: np.nan}), ("FLT_MAX pair", {33: FMAX, 34: FMAX}),
                     ("-FLT_MAX pair", {50: -FMAX, 51: -FMAX})):
        d = base.copy()
        for i, x in at.items():
            d[i] = x
        out[name] = d
    pairs = base.copy()
    pairs[1::2] = -pairs[0::2][: len(pairs[1::2])]   # x, -x: every other edge sums to +0
    out["x,-x"] = pairs
    return out


@gpu
def test_projection_of_special_values_equals_the_oracle():
    v, star, start, rec, delta = _line(64, 5)
    with _context(v, star, [start], delta) as ctx:
        tt = ctx.get_tt(0)
        nodes, length, status, _ = oracle_rays(v, tt, star, start, rec, delta=delta)
        with ctx.freeze_rays(rec) as rs:
            for name, d in _special_perturbations(64, np.random.default_rng(7)).items():
                want = oracle_project(d, nodes, length, status, delta)
                pd = ctx.ray_project(d, rec)
                assert _nan_or_bits_equal(pd.values[0], want), f"{name}: {pd.values[0]} != {want}"
                assert _bits_equal(rs.project(d).values, pd.values), f"{name}: ray set, NaN bits included"
                if name in ("+0", "-0", "+-0"):
                    assert (pd.values.view(np.uint32) == 0).all(), name
                if name in ("FLT_MAX pair", "+INF"):
                    assert np.isinf(pd.values).any() and np.isfinite(pd.values).any(), name
                if name in ("NaN", "+INF,-INF"):
                    assert np.isnan(pd.values).any() and not np.isnan(pd.values[0, :7]).any(), name


# ---- GPU: ray sets frozen in many chunks -------------------------------------------------------

def _max_nodes_for_chunk(chunk):
    """The max_nodes whose freeze chunk, STAGING / (2 max_nodes) rays, is exactly `chunk`."""
    m = (STAGING // 2) // chunk
    assert (STAGING // (2 * m)) == chunk and chunk * 2 * m <= STAGING
    return m


def _assert_sets_equal(a, b, d, w, what):
    assert (a.status == b.status).all() and (a.length == b.length).all() and _bits_equal(a.tt, b.tt), what
    pa, pb = a.paths(), b.paths()
    assert (pa[0] == pb[0]).all() and (pa[1] == pb[1]).all(), f"{what}: paths"
    assert _bits_equal(a.project(d).values, b.project(d).values), f"{what}: projection"
    ga, gb = a.backproject(w), b.backproject(w)
    assert ga.quantum_exp == gb.quantum_exp and _bits_equal(ga.grad, gb.grad), f"{what}: back-projection"


@gpu
def test_freezes_in_many_chunks_equal_one_chunk_and_the_oracle():
    """hetero_818, three sources, every third node, stepped three rounds from the start so that rays of every status are
    present: chunks of 2237 rays (prime) and one chunk; the table, paths and operators against the oracle."""
    ms = _golden_cases()["hetero_818"]
    dims = tuple(ms[0]["dims"])
    rec = all_nodes(dims)[::3]
    star = W.star("818")
    ctx, v = _ctx(ms, put=True)
    with ctx:
        ctx.reset()
        ctx.step(3)
        fields = [ctx.get_tt(s) for s in range(3)]
        one_cap = 256                          # STAGING / (2 * 256) > 3 * 11000 rays: one chunk
        assert STAGING // (2 * one_cap) >= 3 * len(rec)
        rays = [oracle_rays(v, f, star, m["start"], rec, max_nodes=one_cap)[:3] for f, m in zip(fields, ms)]
        status = np.stack([r[2] for r in rays])
        assert (status == OK).any() and (status == UNREACHED).any() and (status > UNREACHED).any(), np.bincount(
            status.ravel())
        d = np.random.default_rng(8).standard_normal(dims).astype(F)
        w = _weights(status.shape, 9)
        with ctx.freeze_rays(rec, max_nodes=one_cap) as one, \
                ctx.freeze_rays(rec, max_nodes=_max_nodes_for_chunk(2237)) as many:
            assert many.stats.kernel_launches >= 15 and one.stats.kernel_launches == 2
            assert not (one.status == TRUNCATED).any() and not (many.status == TRUNCATED).any()
            _assert_sets_equal(many, one, d, w, "2237-ray chunks")
            assert (one.status == status).all() and (one.length == np.stack([r[1] for r in rays])).all()
            assert _bits_equal(one.tt, np.stack([f[tuple(rec.T)] for f in fields]))
            offsets, nodes = one.paths()
            want = np.concatenate([r[0][q, :r[1][q]] for r in rays for q in range(len(rec)) if r[2][q] == OK])
            assert (nodes == want).all()
            for s, r in enumerate(rays):
                assert _nan_or_bits_equal(one.project(d).values[s], oracle_project(d, *r)), f"source {s}: projection"
            g, e = oracle_backproject(dims, rays, w, _hd_max("818"))
            sb = many.backproject(w)
            assert sb.quantum_exp == e and _bits_equal(sb.grad, g)
        few = rec[::500]
        wf = _weights((3, len(few)), 10)
        with ctx.freeze_rays(few, max_nodes=(1 << 26) + 1) as single, ctx.freeze_rays(few, max_nodes=one_cap) as ref:
            assert STAGING // (2 * ((1 << 26) + 1)) == 1 and single.stats.kernel_launches >= 3 * len(few)
            _assert_sets_equal(single, ref, d, wf, "one-ray chunks")


@gpu
def test_freeze_with_chunks_that_hold_no_ok_ray():
    """A line whose far part is +INF: the receivers list 150 reachable nodes, 5000 unreachable ones, the 150 again;
    with chunks of 2237 rays the middle chunk has no OK ray."""
    v, star, start, _, delta = _line(200, 11)
    v[150:] = np.inf
    rec = np.array([(x, 0, 0) for x in range(150)] + [(199, 0, 0)] * 5000 + [(x, 0, 0) for x in range(150)], np.int32)
    with _context(v, star, [start], delta) as ctx:
        nodes, length, status, ttr = oracle_rays(v, ctx.get_tt(0), star, start, rec, max_nodes=300)
        assert (status[150:5150] == UNREACHED).all() and (status[:150] == OK).all()
        d = np.random.default_rng(12).standard_normal(v.shape).astype(F)
        w = _weights((1, len(rec)), 13)
        with ctx.freeze_rays(rec, max_nodes=300) as one, \
                ctx.freeze_rays(rec, max_nodes=_max_nodes_for_chunk(2237)) as many:
            assert one.stats.kernel_launches == 2 and many.stats.kernel_launches == 3 + 2   # 3 traces, 2 packings
            _assert_sets_equal(many, one, d, w, "empty chunk")
            assert (many.status[0] == status).all() and (many.length[0] == length).all()
            assert _nan_or_bits_equal(many.project(d).values[0], oracle_project(d, nodes, length, status))
            g, e = oracle_backproject(v.shape, [(nodes, length, status)], w, _hd_max(star))
            sb = many.backproject(w)
            assert sb.quantum_exp == e and _bits_equal(sb.grad, g)


# ---- GPU: location -----------------------------------------------------------------------------

def _station_context(n, dims=(7, 5, 3), seed=1, delta=10.0, v=None):
    """n stations on a small box (several share a node): n fields, cheap to solve."""
    v = W.random_field(dims, seed=seed) if v is None else v
    starts = np.stack(np.unravel_index(np.arange(n) % int(np.prod(dims)), dims), 1).astype(np.int32)
    ctx = P.SweepContext()
    ctx.set_model(v); ctx.set_star(W.star("5"), delta); ctx.set_sources(starts)
    ctx.run()
    return ctx


def _random_events(fields, n, rng, nan_frac=0.3):
    S = fields.shape[0]
    flat = fields.reshape(S, -1)
    at = rng.integers(flat.shape[1], size=n)
    picks = (flat[:, at].T + rng.uniform(0, 20, (n, 1)) + rng.normal(0, 0.5, (n, S))).astype(F)
    picks[rng.random((n, S)) < nan_frac] = np.nan
    return picks


@gpu
def test_origin_times_equal_numpy_division_for_every_pick_count():
    """2 x 904 events, k = 1 .. 904 picks each (twice), on the largest accepted number of stations: every origin
    time is numpy's a / k."""
    S = LOC_MAX_STATIONS
    rng = np.random.default_rng(30)
    with _station_context(S) as ctx:
        fields = _fields(ctx)
        picks = _random_events(fields, 2 * S, rng, nan_frac=0)
        for e in range(2 * S):
            k = e % S + 1
            picks[e, rng.permutation(S)[k:]] = np.nan
        loc = ctx.locate_events(picks)
        want = oracle_locate(fields, picks)
        assert_locations_equal(loc, want, f"k = 1..{S}")
        assert sorted(set(loc.npicks)) == list(range(1, S + 1))


@gpu
def test_location_on_both_sides_of_each_kernel_shape_and_the_station_limit(monkeypatch):
    """Station counts around the switches from 4 to 2 to 1 nodes per thread and the limit, 70 events each in launches
    of 37 events, on 105 nodes (not a multiple of 32 NB); one-pick events tie over every node, across CTAs."""
    counts = (225, 226, 452, 453, LOC_MAX_STATIONS)
    rng = np.random.default_rng(31)
    monkeypatch.setenv("SWEEPTT_LOCATE_CHUNK", "37")
    with _station_context(LOC_MAX_STATIONS + 20) as ctx:
        fields = _fields(ctx)
        accepted = []
        for m in range(LOC_MAX_STATIONS - 4, LOC_MAX_STATIONS + 5):
            try:
                ctx.locate_events(np.full((1, m), 5, F), sources=(0, m))
                accepted.append(m)
            except P.SweepError as err:
                assert "shared memory" in str(err)
        largest = max(accepted, default=None)
        assert largest == LOC_MAX_STATIONS, f"largest accepted station count: {largest}"
        assert accepted == list(range(LOC_MAX_STATIONS - 4, largest + 1))
        for m in counts:
            picks = _random_events(fields[:m], 70, rng)
            for e in range(6):   # one pick: every node fits exactly, the first node wins
                picks[e] = np.nan
                picks[e, rng.integers(m)] = F(rng.uniform(0, 50))
            loc = ctx.locate_events(picks, sources=(0, m))
            assert loc.stats.kernel_launches == 2 + 1
            assert_locations_equal(loc, oracle_locate(fields[:m], picks), f"{m} stations")
            assert (loc.node[:6] == 0).all()


@gpu
def test_location_of_overflowing_misfits_ranks_before_excluded_nodes():
    """Picks of +-3e38 make every misfit overflow float32 to +INF; the event is still located (OK, misfit +INF), at
    the first node that is not excluded, ahead of the excluded nodes (+INF slowness) before it."""
    dims = (9, 6, 5)
    v = W.random_field(dims, seed=14)
    v[0, :, :] = np.inf   # nodes 0 .. 29: +INF time at every station, excluded
    v[4, 2, 1] = np.inf
    starts = np.array([(3, 1, 1), (8, 5, 4), (5, 0, 0), (6, 3, 2), (1, 5, 4), (7, 0, 3)], np.int32)
    ctx = P.SweepContext()
    with ctx:
        ctx.set_model(v); ctx.set_star(W.star("5")); ctx.set_sources(starts)
        ctx.run()
        fields = _fields(ctx)
        picks = np.array([[3e38, -3e38, 3e38, -3e38, 1.0, np.nan],
                          [-3e38, np.nan, np.nan, 3e38, np.nan, np.nan],
                          [3e38, 2.0, 5.0, np.nan, 7.0, 1.0],          # mixed: one huge residual
                          [FMAX, -FMAX, FMAX, -FMAX, FMAX, -FMAX]], F)
        loc = ctx.locate_events(picks)
        assert_locations_equal(loc, oracle_locate(fields, picks), "overflow")
        assert (loc.status == api.LOC_OK).all() and (loc.misfit == np.inf).all()
        assert (np.ravel_multi_index(tuple(loc.node.T), dims) == int(np.prod(dims[1:]))).all()   # node (1, 0, 0)
        for p in picks:
            box = ctx.misfit_box(p)
            assert (_bits32(box) == _bits32(oracle_misfit(fields, p)[0])).all()


@gpu
def test_location_with_subnormal_misfits_and_signed_zero_picks():
    """delta = 1e-18: times near 1e-17, picks off by about 1e-20, so misfits are float32 subnormals; -0.0 and +0.0
    picks; an all-NaN row gives a misfit box of +0 everywhere."""
    dims = (8, 7, 6)
    rng = np.random.default_rng(15)
    with _station_context(7, dims, seed=16, delta=1e-18) as ctx:
        fields = _fields(ctx)
        flat = fields.reshape(7, -1)
        at = rng.integers(flat.shape[1], size=40)
        picks = (flat[:, at].T + rng.normal(0, 3e-21, (40, 7))).astype(F)
        picks[rng.random(picks.shape) < 0.2] = np.nan
        zeros = rng.choice(np.array([0.0, -0.0], F), (8, 7))
        picks = np.concatenate([picks, zeros])
        loc = ctx.locate_events(picks)
        assert_locations_equal(loc, oracle_locate(fields, picks), "subnormal / signed zero")
        sub = (loc.misfit > 0) & (loc.misfit < 2.0 ** -126)
        assert sub.sum() >= 10, loc.misfit
        for p in (picks[0], picks[-1], picks[-2]):
            assert (_bits32(ctx.misfit_box(p)) == _bits32(oracle_misfit(fields, p)[0])).all()
        none = ctx.misfit_box(np.full(7, np.nan, F))
        assert (none.view(np.uint32) == 0).all(), "no pick: every node's misfit is +0"


# ---- GPU: put_tt input -------------------------------------------------------------------------

@gpu
def test_put_tt_refuses_nan_and_negative_times_and_leaves_the_context_as_it_was():
    ms = _golden_cases()["rand_818"]
    dims = tuple(ms[0]["dims"])
    ctx, v = _ctx(ms, put=True)
    with ctx:
        before = [ctx.get_tt(s) for s in range(ctx.nsrc)]
        pool = ctx.pool_bytes
        for value, name, at in ((np.nan, "NaN", 17), (-1.0, "negative", 0), (-np.inf, "-INF", 500),
                                (-0.0, "-0.0", 3), (-TINY, "negative", int(np.prod(dims)) - 1)):
            bad = ms[1]["tt"].copy()
            bad.ravel()[at] = value
            with pytest.raises(P.SweepError, match=rf"tt\[{at}\] of source 1 is {name}"):
                ctx.put_tt(1, bad)
            assert ctx.pool_bytes == pool
            for s in range(ctx.nsrc):
                assert _bits_equal(ctx.get_tt(s), before[s]), (name, s)
        # +INF is an upper bound like any other: from a field that is +INF but at the start, stepping converges
        # to the golden field
        up = np.full(dims, np.inf, F)
        up[tuple(ms[1]["start"])] = 0
        ctx.put_tt(1, up)
        for _ in range(1000):
            changed, _ = ctx.step(1)
            if not changed:
                break
        assert _bits_equal(ctx.get_tt(1), ms[1]["tt"]) and _bits_equal(ctx.get_tt(0), before[0])
