"""The LSQR step of a ray set (include/sweeptt.h, sweeptt_rayset_lsqr; DESIGN §3.11) at the boundaries of its fixed-order
reduction, on boxes with unit axes, at the float edges of every accepted input, and on the inputs whose norms overflow.

The yardstick is lsqr_restated of test_rayset_lsqr.py (scipy's lsqr statement for statement, every norm sqrt(sumsq)),
applying G through the set's own operators (set_operator) or the CPU oracle; every device result must equal it bit
for bit in x, istop, itn and the six norms.
CPU: the restatement (and scipy on the explicit matrix) turns x into NaN on a b whose sum of squares overflows and on
a smooth whose D rows overflow, which is why the device refuses them; a b whose squares underflow is b = 0 there too;
the sizes below do sit on the reduction's block boundaries.
GPU (-m gpu): u of length m = 1 .. 4097 on lines of 2047, 2048 and 2049 nodes; u of length 2048^2 - 1, 2048^2 and
2048^2 + 1 (a 1448 x 1448 x 1 slab with smoothing: a second and a third reduction level); v and x of length 2048^2 and
2048^2 + 2048; each under SWEEPTT_LSQR_CTAS = 1, 2, nb - 1, nb, nb + 1; boxes with axes of length 1 under every
SWEEPTT_WINDOW_AXIS; subnormal, tiny, huge and signed-zero b; damp, smooth and delta from the subnormals to overflow;
every option edge; an empty selection; stop reasons 4 and 5; the refusal of the three overflow routes, after which
the set still solves bit for bit and every byte of the workspace is back.  The large boxes get their fields from
put_tt, which also runs once in a fresh process on a simple-kernel box of 16,384 tiles.  The GPU tests take 16 s on
one B200 (1000 W power limit)."""
import math
import subprocess
import sys
import textwrap

import numpy as np
import pytest
import torch
from scipy.sparse.linalg import lsqr

import uoparallel_seismic_project_b200 as P
from uoparallel_seismic_project_b200 import api, workloads as W

from conftest import ROOT, make_field
from test_rays import _golden_cases, all_nodes
from test_rayset import explicit_g, oracle_operator
from test_rayset_lsqr import (_golden_problem, _golden_set, assert_same_solution, d_count, d_rows, lsqr_restated,
                              set_operator, sumsq)
from test_tomography import AXIS_STAR, _hd_max, quantum_exp

gpu = pytest.mark.gpu
OK = api.RAY_OK
BLOCK = 2048
SQRT_MAX = math.sqrt(np.finfo(np.float64).max)   # the largest double whose square is finite
SLAB = (1448, 1448, 1)                            # d_count(SLAB) = 2048^2 - 3792


def _solution(s):
    """An LsqrSolution as the tuple lsqr_restated returns, to compare two device solves."""
    return s.x.ravel(), s.istop, s.itn, s.r1norm, s.r2norm, s.anorm, s.acond, s.arnorm, s.xnorm


def _all_nan(x):
    return bool(np.isnan(np.asarray(x)).all())


# ---- CPU ---------------------------------------------------------------------------------------

def test_the_sizes_sit_on_the_reduction_boundaries():
    assert d_count(SLAB) + 3792 == BLOCK * BLOCK
    assert 2049 * 2048 == BLOCK * BLOCK + BLOCK
    # sumsq of 2048^2 + 1 elements takes three levels: 2049 block sums, then 2, then 1
    v = np.zeros(BLOCK * BLOCK + 1)
    v[-1], v[0] = 3.0, 4.0
    assert sumsq(v) == 25.0


def test_restatement_and_scipy_go_nan_when_a_norm_overflows():
    """b with an entry 2^512 (||b||^2 = +inf) and smooth = 1e300 (the D rows of v square to +inf): 1/inf = 0 and
    0 * inf = NaN make x all NaN and every stopping test false, so the loop runs to iter_lim."""
    ms, rays, rows, b = _golden_problem("rand_818")
    dims = tuple(ms[0]["dims"])
    op = oracle_operator(dims, rays, rows, _hd_max(ms[0]["star"]))
    big = b.copy()
    big[5] = 2.0 ** 512
    for bb, kw in [(big, {}), (b, dict(smooth=1e300))]:
        out = lsqr_restated(op.matvec, op.rmatvec, bb, dims, iter_lim=3, **kw)
        assert _all_nan(out[0]) and out[1:3] == (7, 3), (kw, out[1:3])
    G = explicit_g(dims, rays, rows)
    with np.errstate(all="ignore"):
        ref = lsqr(G, big, iter_lim=3)
    assert _all_nan(ref[0]) and ref[1:3] == (7, 3)


def test_an_underflowing_b_is_b_zero_as_in_scipy():
    """Every square of 5e-324 rounds to +0, so ||b|| = 0: x = 0, istop = 0, itn = 0 in scipy and the restatement.  A b
    of about 1e-160 has subnormal squares and is solved; scipy's eps in the denominator of test2 stops both after one
    iteration with istop = 2."""
    ms, rays, rows, b = _golden_problem("rand_818")
    dims = tuple(ms[0]["dims"])
    op = oracle_operator(dims, rays, rows, _hd_max(ms[0]["star"]))
    G = explicit_g(dims, rays, rows)
    tiny = np.full(b.size, 5e-324)
    out = lsqr_restated(op.matvec, op.rmatvec, tiny, dims)
    ref = lsqr(G, tiny)
    assert out[1:3] == (0, 0) and ref[1:3] == (0, 0) and not out[0].any() and not ref[0].any()
    sub = b * 1e-160
    assert 0 < sumsq(sub) < np.finfo(np.float64).tiny
    out = lsqr_restated(op.matvec, op.rmatvec, sub, dims, iter_lim=5)
    ref = lsqr(G, sub, iter_lim=5)
    assert out[1:3] == ref[1:3] == (2, 1) and np.isfinite(out[0]).all() and out[0].any()


# ---- GPU helpers -------------------------------------------------------------------------------

def _manhattan_set(dims, start, receivers):
    """A set on a constant box (slowness 0.25, the axis star, delta = 4: every edge takes exactly 1) whose field is
    the exact Manhattan distance to the start, loaded with put_tt: no sweep of the large boxes."""
    v = np.full(dims, 0.25, np.float32)
    grid = np.indices(dims).reshape(3, -1).T
    tt = np.abs(grid - np.asarray(start)).sum(1).astype(np.float32).reshape(dims)
    ctx = P.SweepContext(kernel=api.KERNEL_SIMPLE)
    ctx.set_model(v); ctx.set_star(AXIS_STAR, 4.0); ctx.set_sources([start])
    ctx.put_tt(0, tt)
    rs = ctx.freeze_rays(np.asarray(receivers, np.int32))
    assert (rs.status == OK).all()
    return ctx, rs


@gpu
def test_put_tt_in_a_process_that_prepared_no_tiled_kernel():
    """put_tt folds its marks into the work list with the single-block compaction, whose keys (4 bytes per tile and
    source) need more than the default 48 KB of shared memory above 12,288 tiles.  The attribute that allows it was
    set only when a tiled kernel was prepared, so put_tt on a simple-kernel context of 16,384 tiles failed with
    "invalid argument" in a fresh process.  Run in one, since any tiled context earlier in this one hides it."""
    script = textwrap.dedent(f"""
        import sys
        sys.path.insert(0, {str(ROOT)!r})
        import numpy as np
        import uoparallel_seismic_project_b200 as P
        from uoparallel_seismic_project_b200 import api
        dims = (1024, 1024, 1)
        tt = np.add.outer(np.arange(1024.0), np.arange(1024.0)).astype(np.float32).reshape(dims)
        star = np.array({AXIS_STAR.tolist()}, np.int32)
        with P.SweepContext(kernel=api.KERNEL_SIMPLE) as ctx:
            ctx.set_model(np.full(dims, 0.25, np.float32)); ctx.set_star(star, 4.0); ctx.set_sources([(0, 0, 0)])
            ctx.put_tt(0, tt)
            assert ctx.count_violations(0) == 0 and (ctx.get_tt(0).view(np.uint32) == tt.view(np.uint32)).all()
        print("ok")
    """)
    r = subprocess.run([sys.executable, "-c", script], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and r.stdout.strip() == "ok", (r.stdout, r.stderr[-2000:])


def _square(centre, half):
    cx, cy, cz = centre
    return [(x, y, cz) for x in range(cx - half, cx + half + 1) for y in range(cy - half, cy + half + 1)]


def _first(rs, m):
    """Rows selecting the first m rays of the set."""
    rows = np.zeros(rs.shape, bool)
    rows.ravel()[:m] = True
    return rows


def _check(rs, rows, b, what, iters=(0, 3), **kw):
    """The device solve against the restatement on the set's operators, with iter_lim = 0 (r1norm = ||b||, arnorm =
    alfa beta: the u and v sums alone) and then a few iterations (the xw pass too).  Returns the last solve."""
    matvec, rmatvec = set_operator(rs, rows)
    for it in iters:
        want = lsqr_restated(matvec, rmatvec, b, rs.dims, iter_lim=it, **kw)
        got = rs.lsqr(b, rows, iter_lim=it, **kw)
        assert_same_solution(got, want, f"{what} iter_lim={it}")
        if it == 0:
            assert got.itn == 0 and got.r1norm == np.sqrt(sumsq(b))
    return got


def _grid_independent(rs, rows, b, first, nb, monkeypatch, what, **kw):
    for ctas in (1, 2, nb - 1, nb, nb + 1):
        monkeypatch.setenv("SWEEPTT_LSQR_CTAS", str(ctas))
        assert_same_solution(rs.lsqr(b, rows, **kw), _solution(first), f"{what} ctas={ctas}")
    monkeypatch.delenv("SWEEPTT_LSQR_CTAS")


# ---- GPU: the reduction boundaries -------------------------------------------------------------

@gpu
@pytest.mark.parametrize("n", [2047, 2048, 2049])
def test_u_and_v_sums_at_the_block_boundaries_of_a_line(n):
    """A line of n nodes (v, x of length n) with every node a receiver three times over; the rows select the first m
    rays, m in {1, 2047, 2048, 2049, 4096, 4097} (u of length m, no smoothing)."""
    rec = [(x, 0, 0) for x in range(n)] * 3
    rng = np.random.default_rng(n)
    ctx, rs = _manhattan_set((n, 1, 1), (0, 0, 0), rec)
    with ctx, rs:
        for m in (1, 2047, 2048, 2049, 4096, 4097):
            b = rng.standard_normal(m)
            _check(rs, _first(rs, m), b, f"line {n}, m = {m}", damp=0.5)


@gpu
def test_u_sums_at_the_second_and_third_reduction_levels(monkeypatch):
    """The 1448 x 1448 x 1 slab with smoothing: m + mD = 2048^2 - 1, 2048^2, 2048^2 + 1 (2048 block sums then one; 2049,
    then 2, then 1), and the last under every grid around its 2049 blocks."""
    centre = (724, 724, 0)
    ctx, rs = _manhattan_set(SLAB, centre, _square(centre, 31))
    rng = np.random.default_rng(1448)
    with ctx, rs:
        for m in (3791, 3792, 3793):
            assert m + d_count(SLAB) - BLOCK * BLOCK == m - 3792
            b = rng.standard_normal(m)
            got = _check(rs, _first(rs, m), b, f"slab m = {m}", iters=(0, 2), smooth=2.0, damp=0.5)
        _grid_independent(rs, _first(rs, 3793), b, got, BLOCK + 1, monkeypatch, "slab", iter_lim=2, smooth=2.0,
                          damp=0.5)


@gpu
@pytest.mark.parametrize("dims", [(2048, 2048, 1), (2049, 2048, 1)])
def test_v_and_x_sums_of_a_box_of_2048_squared_nodes(dims, monkeypatch):
    """v and x of length 2048^2 (2048 block sums, one reduction) and 2048^2 + 2048 (2049 block sums, two); the larger
    under every grid around its 2049 blocks."""
    centre = (1024, 1024, 0)
    ctx, rs = _manhattan_set(dims, centre, _square(centre, 3))
    b = np.random.default_rng(dims[0]).standard_normal(rs.status.size)
    rows = rs.status == OK
    with ctx, rs:
        got = _check(rs, rows, b, f"box {dims}", damp=0.5)
        if dims[0] == 2049:
            _grid_independent(rs, rows, b, got, BLOCK + 1, monkeypatch, "box", iter_lim=3, damp=0.5)


# ---- GPU: unit axes ----------------------------------------------------------------------------

@gpu
@pytest.mark.parametrize("axis", ["0", "1", "2"])
@pytest.mark.parametrize("dims", [(1, 1, 1), (9, 1, 1), (1, 9, 1), (1, 1, 9), (1, 5, 7), (3, 2, 1)])
def test_smoothing_on_boxes_with_unit_axes(dims, axis, monkeypatch):
    """Every window axis permutes the kernel axes that lsqr_d_row / lsqr_dt index away from the caller axes of D."""
    monkeypatch.setenv("SWEEPTT_WINDOW_AXIS", axis)
    v = make_field("random", dims, sum(dims))
    with P.SweepContext(kernel=api.KERNEL_SIMPLE) as ctx:
        ctx.set_model(v); ctx.set_star(AXIS_STAR); ctx.set_sources([(0, 0, 0)])
        ctx.run()
        with ctx.freeze_rays(all_nodes(dims)) as rs:
            rows = rs.status == OK
            assert rows.all()
            b = np.random.default_rng(7).standard_normal(int(rows.sum()))
            _check(rs, rows, b, f"{dims} axis {axis}", iters=(0, 12), smooth=1.5, damp=0.25)


# ---- GPU: float edges of accepted inputs -------------------------------------------------------

def _rmatvec_watch(rmatvec, zero_w):
    """rmatvec that records, per call, whether float32(y) is all +-0 (max |W| = 0: the E = 0 branch)."""
    def f(y):
        zero_w.append(not np.float32(y).any())
        return rmatvec(y)
    return f


@gpu
def test_float_edges_of_b_damp_smooth_and_the_options():
    ms, rays, rows, b = _golden_problem("rand_818")
    dims = tuple(ms[0]["dims"])
    rng = np.random.default_rng(9)
    sign = rng.choice([-1.0, 1.0], b.size)
    negz = b.copy()
    negz[::3] = -0.0
    top = b.copy()
    top[0] = SQRT_MAX
    with np.errstate(over="ignore"):
        assert np.isfinite(SQRT_MAX * SQRT_MAX) and np.isinf(np.nextafter(SQRT_MAX, np.inf) ** 2)
    mixed = np.where(rng.random(b.size) < 0.5, 1.0, 1e-50) * sign
    cases = [
        ("b = 5e-324", np.full(b.size, 5e-324), {}),
        ("b ~ 1e-160", b * 1e-160, {}),
        ("b with -0.0", negz, {}),
        ("b all -0.0", np.full(b.size, -0.0), dict(smooth=3.0)),
        ("b = +-1e150", sign * 1e150, dict(damp=1.0)),
        ("b with sqrt(DBL_MAX)", top, {}),
        ("b of 1 and 1e-50", mixed, dict(smooth=1.0)),
        ("damp 5e-324", b, dict(damp=5e-324)),
        ("damp 1e-300", b, dict(damp=1e-300)),
        ("damp^2 finite", b, dict(damp=SQRT_MAX)),
        ("damp^2 overflows", b, dict(damp=float(np.nextafter(SQRT_MAX, np.inf)))),
        ("smooth 5e-324", b, dict(smooth=5e-324)),
        ("smooth 1e-300", b, dict(smooth=1e-300)),
        ("smooth 1e100", b, dict(smooth=1e100)),
        ("atol = btol = 0", b, dict(atol=0.0, btol=0.0)),
        ("conlim 0", b, dict(conlim=0.0, damp=1.0)),
        ("conlim inf", b, dict(conlim=np.inf, damp=1.0)),
        ("iter_lim 0", b, dict(iter_lim=0, smooth=2.0)),
        ("iter_lim 1", b, dict(iter_lim=1, smooth=2.0)),
    ]
    ctx, rs = _golden_set("rand_818")
    with ctx, rs:
        matvec, rmatvec = set_operator(rs, rows)
        for what, bb, kw in cases:
            kw = dict(dict(iter_lim=8), **kw)
            want = lsqr_restated(matvec, rmatvec, bb, dims, **kw)
            got = rs.lsqr(bb, rows, **kw)
            assert_same_solution(got, want, what)
            if what in ("b = 5e-324", "b all -0.0"):
                assert (got.istop, got.itn, got.r1norm) == (0, 0, 0.0) and not got.x.any(), what
            elif kw["iter_lim"]:
                assert got.itn >= 1 and np.isfinite(got.x).all(), what
        unit = rng.standard_normal(dims)
        unit /= np.sqrt(sumsq(unit))   # as LSQR's v: every difference is below 1/2, so 5e-324 times it is +-0
        assert np.abs(np.diff(unit.ravel())).max() < 0.5 and (d_rows(unit, dims, 5e-324) == 0).all()
        # a strong smooth: from the first iteration on, the G rows of u are below float32's range, every W is 0
        tiny, zero_w = b * 1e-30, []
        kw = dict(smooth=1e60, atol=0.0, btol=0.0, conlim=0.0, iter_lim=4)
        want = lsqr_restated(matvec, _rmatvec_watch(rmatvec, zero_w), tiny, dims, **kw)
        assert len(zero_w) >= 2 and not zero_w[0] and all(zero_w[1:]), zero_w
        assert_same_solution(rs.lsqr(tiny, rows, **kw), want, "smooth 1e60, W = 0")
        # no row selected: u is empty, or only the D rows (zero); x = 0
        none = np.zeros(rs.shape, bool)
        for smooth in (0.0, 3.0):
            got = rs.lsqr(np.zeros(0), none, smooth=smooth, damp=1.0)
            want = lsqr_restated(*set_operator(rs, none), np.zeros(0), dims, smooth=smooth, damp=1.0)
            assert_same_solution(got, want, f"m = 0, smooth {smooth}")
            assert (got.istop, got.itn) == (0, 0) and not got.x.any()


@gpu
@pytest.mark.parametrize("delta", [1e-20, 1e20])
def test_delta_at_both_ends_of_the_quantum_exponent(delta):
    ms = _golden_cases()["rand_818"]
    dims = tuple(ms[0]["dims"])
    v = make_field(ms[0]["kind"], dims, ms[0]["seed"])
    star = W.star(ms[0]["star"])
    with P.SweepContext() as ctx:
        ctx.set_model(v); ctx.set_star(star, delta); ctx.set_sources([m["start"] for m in ms])
        ctx.run()
        with ctx.freeze_rays(all_nodes(dims)) as rs:
            rows = rs.status == OK
            b = np.random.default_rng(3).standard_normal(int(rows.sum())) * delta
            w = np.zeros(rs.shape, np.float32)
            w[rows] = b / np.sqrt(sumsq(b))
            e = rs.backproject(w).quantum_exp
            assert e == quantum_exp(_hd_max(star, delta), float(np.abs(w).max()), w.size)
            assert (e < -100) if delta < 1 else (e > 10), e
            for kw in (dict(damp=0.0), dict(damp=1e-3 * delta, smooth=delta)):
                want = lsqr_restated(*set_operator(rs, rows), b, dims, iter_lim=10, **kw)
                assert_same_solution(rs.lsqr(b, rows, iter_lim=10, **kw), want, f"delta {delta} {kw}")


def _line_set(ctx, n, rec):
    v = np.random.default_rng(1).uniform(0.2, 0.4, (n, 1, 1)).astype(np.float32)
    ctx.set_model(v); ctx.set_star(AXIS_STAR); ctx.set_sources([(0, 0, 0)])
    ctx.run()
    return ctx.freeze_rays(np.array([(x, 0, 0) for x in rec], np.int32))


@gpu
def test_stop_reasons_4_and_5():
    """4: a consistent system (b = G x_true on a line of 4 nodes, 3 rays), atol = btol = 0, where the estimate of
    ||r|| keeps shrinking after convergence.  5: an inconsistent one (two rays twice with other times, damp 0.5),
    where the estimate of ||A^T r|| does.  6 (cond(A) >= 1/eps) is not reached: the golden sets keep acond near 1e4
    after 600 iterations, and a ray set's G has no tunable condition number."""
    with P.SweepContext(kernel=api.KERNEL_SIMPLE) as ctx:
        with _line_set(ctx, 4, [1, 2, 3]) as rs:
            rows = rs.status == OK
            matvec, rmatvec = set_operator(rs, rows)
            b = matvec(np.array([0.3, -1.2, 0.7, 2.0]))
            want = lsqr_restated(matvec, rmatvec, b, rs.dims, atol=0.0, btol=0.0, conlim=0.0, iter_lim=50)
            assert want[1] == 4, want[1:3]
            assert_same_solution(rs.lsqr(b, rows, atol=0.0, btol=0.0, conlim=0.0, iter_lim=50), want, "istop 4")
        with _line_set(ctx, 3, [1, 2, 1, 2]) as rs:
            rows = rs.status == OK
            b = np.array([1.0, 2.0, 1.5, 2.5])
            kw = dict(damp=0.5, atol=0.0, btol=0.0, conlim=0.0, iter_lim=50)
            want = lsqr_restated(*set_operator(rs, rows), b, rs.dims, **kw)
            assert want[1] == 5, want[1:3]
            assert_same_solution(rs.lsqr(b, rows, **kw), want, "istop 5")


# ---- GPU: norms that overflow are refused ------------------------------------------------------

@gpu
def test_norms_that_overflow_are_refused_and_leave_the_set_working():
    """A b entry of 2^512 (bnorm = +inf) and a smooth of 1e300 (beta of iteration 1: the D rows of v square to +inf)
    each make the restatement's x all NaN; the device refuses both, leaves x_out and info untouched, frees its
    workspace, and solves the golden problem bit for bit afterwards.  iter_lim is small so that a call which does not
    refuse returns quickly."""
    ms, rays, rows, b = _golden_problem("rand_818")
    dims = tuple(ms[0]["dims"])
    big = b.copy()
    big[5] = 2.0 ** 512
    ctx, rs = _golden_set("rand_818")
    with ctx, rs:
        matvec, rmatvec = set_operator(rs, rows)
        want = rs.lsqr(b, rows, damp=1.0, smooth=1.0, iter_lim=5)   # every kernel loaded before the memory is read
        torch.cuda.synchronize()
        free0 = torch.cuda.mem_get_info()[0]
        for bb, kw, msg in [(big, {}, "‖b‖² overflows"),
                            (b, dict(smooth=1e300), r"beta = ‖u‖ is not finite \(inf\) at iteration 1")]:
            assert _all_nan(lsqr_restated(matvec, rmatvec, bb, dims, iter_lim=3, **kw)[0])
            with pytest.raises(P.SweepError, match=msg):
                rs.lsqr(bb, rows, iter_lim=3, **kw)
        lib = api.load_library()
        opts = api._LsqrOpts(api.C.sizeof(api._LsqrOpts), 0.0, 1e300, 1e-6, 1e-6, 1e8, 3)
        info = api._LsqrInfo(api.C.sizeof(api._LsqrInfo), -5, -5)
        sel = np.ascontiguousarray(rows, np.uint8)
        x = np.full(dims, 7.0)
        assert not lib.sweeptt_rayset_lsqr(rs._h, sel.ctypes.data, b.ctypes.data, api.C.byref(opts), x.ctypes.data,
                                           api.C.byref(info), None)
        assert "beta" in lib.sweeptt_last_error().decode()
        assert (x == 7.0).all() and (info.istop, info.itn) == (-5, -5), "x_out and info are untouched"
        after = rs.lsqr(b, rows, damp=1.0, smooth=1.0, iter_lim=5)
        torch.cuda.synchronize()
        free1 = torch.cuda.mem_get_info()[0]
        assert_same_solution(after, _solution(want), "after the refusals")
        assert_same_solution(after, lsqr_restated(matvec, rmatvec, b, dims, damp=1.0, smooth=1.0, iter_lim=5),
                             "the restatement")
    assert free1 == free0, (free0, free1)


@gpu
def test_a_projection_that_overflows_is_refused():
    """A line of 51 nodes with delta = 1e38 and one ray over all of it: the back-projection of W = 1 is at most
    2 hd = 1e38 per node, but the float32 projection of the normalised v overflows, so beta of iteration 1 is +inf.
    (The restatement cannot go on from there: u = 0 * inf is NaN, and the set's back-projection refuses NaN
    weights.)"""
    n = 51
    v = np.full((n, 1, 1), 1e-3, np.float32)
    with P.SweepContext(kernel=api.KERNEL_SIMPLE) as ctx:
        ctx.set_model(v); ctx.set_star(AXIS_STAR, 1e38); ctx.set_sources([(0, 0, 0)])
        ctx.run()
        with ctx.freeze_rays(np.array([(n - 1, 0, 0)], np.int32)) as rs:
            assert (rs.status == OK).all()
            one = np.ones(1)
            matvec, rmatvec = set_operator(rs, rs.status == OK)
            g = rmatvec(one)
            assert np.isfinite(g).all()
            with np.errstate(over="ignore"):
                assert np.isinf(matvec(g / np.sqrt(sumsq(g)))).all()
            with pytest.raises(P.SweepError, match=r"beta = ‖u‖ is not finite \(inf\) at iteration 1"):
                rs.lsqr(one, iter_lim=3)
            x = rs.lsqr(one, iter_lim=0)
            assert (x.istop, x.itn) == (0, 0) and not x.x.any()
