"""The region of every event under a misfit level, summarised on the device (include/sweeptt.h, sweeptt_misfit_regions;
SweepContext.misfit_regions, location_uncertainty).

The yardstick is the misfit box, which tests/test_locate.py pins bit for bit against oracle_misfit: here the region is
restated in numpy as R = box <= level, followed by integer sums and min / max, with the oracle's t0 for the origin-time
range.  CPU: a C99 client, the kernel never fuses a multiply-add, mean() / covariance() against Fraction arithmetic,
the levels of location_uncertainty.  GPU (-m gpu): every output bit for bit on random, heterogeneous and contrast
models under both kernels, every axis permutation and put_tt; the levels 0, the best misfit and its float32
neighbours, NaN, above every finite misfit, -0.0; refused levels that leave the context as it was; overflowing misfits
and unreachable events; chunking, repeats and source ranges; the station counts around each kernel shape and the
limit; the moment-overflow refusal; the one-shot call; full-size config 3."""
import re
import shutil
import subprocess
from fractions import Fraction

import numpy as np
import pytest
import torch

import uoparallel_seismic_project_b200 as P
from uoparallel_seismic_project_b200 import api, workloads as W

from conftest import ROOT, make_field
from test_locate import _bits32, _bits64, _context, _events, _fields, _stations, oracle_misfit
from test_operator_edges import LOC_MAX_STATIONS, _random_events, _station_context

gpu = pytest.mark.gpu
F = np.float32
FMAX = np.finfo(F).max
DIMS = (21, 18, 16)


# ---- the restatement ---------------------------------------------------------------------------

def oracle_regions(fields, picks, levels):
    """(count, lo, hi, moments, origin_min, origin_max, status) of R_e = box_e <= levels[e] for every event."""
    E = len(picks)
    count = np.zeros(E, np.int64)
    lo = np.full((E, 3), -1, np.int32)
    hi = np.full((E, 3), -1, np.int32)
    moments = np.zeros((E, 9), np.int64)
    omin = np.full(E, np.nan)
    omax = np.full(E, np.nan)
    status = np.zeros(E, np.int32)
    for e, p in enumerate(picks):
        mis, t0, k, excl = oracle_misfit(fields, p)
        status[e] = api.LOC_NO_PICKS if k == 0 else api.LOC_UNREACHED if excl.all() else api.LOC_OK
        if k == 0 or np.isnan(levels[e]):
            continue
        R = mis <= F(levels[e])
        c = np.argwhere(R).astype(np.int64)
        count[e] = len(c)
        if not len(c):
            continue
        lo[e], hi[e] = c.min(0), c.max(0)
        moments[e] = [c[:, 0].sum(), c[:, 1].sum(), c[:, 2].sum(), (c[:, 0] ** 2).sum(), (c[:, 1] ** 2).sum(),
                      (c[:, 2] ** 2).sum(), (c[:, 0] * c[:, 1]).sum(), (c[:, 0] * c[:, 2]).sum(),
                      (c[:, 1] * c[:, 2]).sum()]
        omin[e], omax[e] = t0[R].min(), t0[R].max()
    return count, lo, hi, moments, omin, omax, status


def assert_regions_equal(got, want, what):
    count, lo, hi, moments, omin, omax, status = want
    assert (got.status == status).all(), f"{what}: status {got.status} != {status}"
    bad = np.nonzero(got.count != count)[0]
    assert not len(bad), f"{what}: counts differ for events {bad}: {got.count[bad]} != {count[bad]}"
    assert (got.lo == lo).all() and (got.hi == hi).all(), f"{what}: bounding box"
    assert (got.moments == moments).all(), f"{what}: moments"
    assert (_bits64(got.origin_min) == _bits64(omin)).all(), f"{what}: origin min"
    assert (_bits64(got.origin_max) == _bits64(omax)).all(), f"{what}: origin max"


def assert_same_regions(a, b, what):
    for f in ("count", "lo", "hi", "moments", "npicks", "status"):
        assert (getattr(a, f) == getattr(b, f)).all(), f"{what}: {f}"
    for f in ("origin_min", "origin_max"):
        assert (_bits64(getattr(a, f)) == _bits64(getattr(b, f))).all(), f"{what}: {f}"


def _concat(parts):
    fields = ("count", "lo", "hi", "moments", "origin_min", "origin_max", "npicks", "status")
    return api.MisfitRegions(*(np.concatenate([getattr(x, f) for x in parts]) for f in fields), None)


def _quantile_levels(fields, picks, seed):
    """A level per event between its best misfit and well above it (quantiles of its finite misfits)."""
    rng = np.random.default_rng(seed)
    levels = np.empty(len(picks), F)
    for e, p in enumerate(picks):
        mis = oracle_misfit(fields, p)[0]
        fin = mis[np.isfinite(mis)]
        levels[e] = F(np.quantile(fin, rng.choice([0.0, 0.001, 0.01, 0.1, 0.5]))) if len(fin) else F(1)
    return levels


# ---- CPU ---------------------------------------------------------------------------------------

@pytest.mark.skipif(shutil.which("cuobjdump") is None, reason="cuobjdump not on PATH")
def test_region_kernel_never_fuses_multiply_add():
    out = subprocess.run(["cuobjdump", "-sass", str(P.lib_path())], capture_output=True, text=True, check=True).stdout
    funcs, name = {}, None
    for line in out.splitlines():
        mm = re.search(r"Function : (\S+)", line)
        if mm:
            name = mm.group(1)
            funcs[name] = []
        elif name and re.match(r"\s+/\*[0-9a-f]{4,6}\*/", line):
            funcs[name].append(line)
    kernels = {k: v for k, v in funcs.items() if "region_kernel" in k}
    assert len(kernels) == 3, sorted(kernels)   # region_kernel<4, 2, 1>
    for k, lines in kernels.items():
        text = "\n".join(lines)
        assert "DADD" in text and "DMUL" in text, k
        assert not re.search(r"\b[DF]FMA2?\b", text), f"{k}: fused multiply-add found"


def test_c99_client_calls_misfit_regions(tmp_path):
    """A strict C99 client compiles and links.  Without a GPU the call fails with "null context"; with one, a 4x4x4
    box and one station: one pick makes every node fit exactly, so level 0 gives the whole box."""
    src = tmp_path / "client.c"
    src.write_text(r'''
#include <stdio.h>
#include "sweeptt.h"
int main(void) {
  struct FS fs[7] = {{1, 0, 0, 0.f}, {-1, 0, 0, 0.f}, {0, 1, 0, 0.f}, {0, -1, 0, 0.f}, {0, 0, 1, 0.f},
                     {0, 0, -1, 0.f}, {1, 1, 1, 0.f}};
  struct START st[1] = {{0, 0, 0}};
  float v[64], picks[1] = {30.f}, levels[1] = {0.f};
  int64_t count[1], moments[9];
  int32_t bbox[6], status[1];
  double origin[2];
  int i;
  sweeptt_stats stats;
  sweeptt_ctx *ctx;
  for (i = 0; i < 64; i++) v[i] = 1.f;
  sweeptt_star_fill_distances(fs, 7, 10.0f);
  ctx = sweeptt_create(NULL);
  if (!ctx) {
    if (sweeptt_misfit_regions(NULL, 0, 1, picks, 1, levels, count, bbox, moments, origin, status, &stats)) return 2;
    printf("%s\n", sweeptt_last_error());
    return 0;
  }
  if (!sweeptt_set_model(ctx, v, 4, 4, 4) || !sweeptt_set_star(ctx, fs, 7) || !sweeptt_set_sources(ctx, st, 1) ||
      !sweeptt_run(ctx, NULL) ||
      !sweeptt_misfit_regions(ctx, 0, 1, picks, 1, levels, count, bbox, moments, origin, status, &stats)) {
    printf("%s\n", sweeptt_last_error());
    return 3;
  }
  sweeptt_destroy(ctx);
  if (status[0] != SWEEPTT_LOC_OK || count[0] != 64) return 4;
  for (i = 0; i < 3; i++)
    if (bbox[i] != 0 || bbox[3 + i] != 3 || moments[i] != 96 || moments[3 + i] != 224) return 5;
  if (moments[6] != 144 || moments[7] != 144 || moments[8] != 144 || origin[1] != 30.0 || !(origin[0] < 30.0)) return 6;
  printf("ok\n");
  return 0;
}
''')
    exe = tmp_path / "client"
    lib = P.lib_path()
    subprocess.run(["gcc", "-std=c99", "-pedantic", "-Wall", "-Werror", f"-I{ROOT / 'include'}", "-o", str(exe), str(src),
                    f"-L{lib.parent}", "-lsweeptt", f"-Wl,-rpath,{lib.parent}"], check=True)
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, (r.returncode, r.stdout, r.stderr)
    if torch.cuda.is_available():
        assert "ok" in r.stdout
    else:
        assert r.stdout.count("null context") == 1, r.stdout


def _regions_from_moments(count, moments):
    E = len(count)
    return api.MisfitRegions(np.asarray(count, np.int64), np.zeros((E, 3), np.int32), np.zeros((E, 3), np.int32),
                             np.asarray(moments, np.int64).reshape(E, 9), np.zeros(E), np.zeros(E),
                             np.zeros(E, np.int32), np.zeros(E, np.int32), None)


def test_mean_and_covariance_are_the_exact_quotients_rounded_once():
    rng = np.random.default_rng(40)
    sets = [np.array([[5, 7, 11]]),                                       # count 1: zero covariance
            np.array([[0, 0, 0], [1, 2, 3]]),
            rng.integers(0, 2401, (1000, 3)),
            rng.integers(0, 3, (7, 3)),
            np.array([[2400, 2400, 500]] * 3 + [[0, 0, 0]])]
    count, moments = [], []
    for c in sets:
        c = c.astype(np.int64)
        count.append(len(c))
        moments.append([c[:, 0].sum(), c[:, 1].sum(), c[:, 2].sum(), (c[:, 0] ** 2).sum(), (c[:, 1] ** 2).sum(),
                        (c[:, 2] ** 2).sum(), (c[:, 0] * c[:, 1]).sum(), (c[:, 0] * c[:, 2]).sum(),
                        (c[:, 1] * c[:, 2]).sum()])
    count.append(0)
    moments.append([0] * 9)
    reg = _regions_from_moments(count, moments)
    mean, cov = reg.mean(), reg.covariance()
    assert mean.shape == (len(count), 3) and cov.shape == (len(count), 3, 3)
    for e, c in enumerate(sets):
        n = len(c)
        for a in range(3):
            want = Fraction(int(c[:, a].sum()), n)
            assert mean[e, a] == float(want)
            for b in range(3):
                ca, cb = [Fraction(int(x)) for x in c[:, a]], [Fraction(int(x)) for x in c[:, b]]
                ma, mb = sum(ca) / n, sum(cb) / n
                want = sum((x - ma) * (y - mb) for x, y in zip(ca, cb)) / n
                assert cov[e, a, b] == float(want), (e, a, b)
    assert (cov[0] == 0).all() and (mean[0] == [5, 7, 11]).all()
    assert np.isnan(mean[-1]).all() and np.isnan(cov[-1]).all()
    assert np.allclose(cov[2], np.cov(sets[2].T, bias=True), rtol=1e-12)


def test_uncertainty_levels():
    from scipy.stats import chi2
    misfit = np.array([0.5, 0.0, np.inf, np.inf, 3e38, 1.25], F)
    status = np.array([api.LOC_OK, api.LOC_OK, api.LOC_NO_PICKS, api.LOC_OK, api.LOC_OK, api.LOC_UNREACHED], np.int32)
    loc = api.Locations(np.zeros((6, 3), np.int32), misfit, np.zeros(6), np.ones(6, np.int32), status, None)
    sigma = np.array([0.1, 2.0, 1.0, 1.0, 1e19, 1.0])
    lv = P.uncertainty_levels(loc, sigma, 0.9)
    q = chi2.ppf(0.9, 3)
    assert lv.dtype == F
    assert lv[0] == F(np.float64(F(0.5)) + 0.1 * 0.1 * q) and lv[1] == F(4.0 * q)
    assert np.isnan(lv[[2, 3, 5]]).all()          # not OK, or an overflowing best misfit: no region
    assert lv[4] == FMAX                          # beyond float32: every finite misfit is inside
    assert P.uncertainty_levels(loc, 0.5)[1] == F(0.25 * chi2.ppf(0.95, 3))
    for bad in (0.0, -1.0, np.inf, np.nan):
        with pytest.raises(P.SweepError, match="sigma"):
            P.uncertainty_levels(loc, bad)
    with pytest.raises(P.SweepError, match="confidence"):
        P.uncertainty_levels(loc, 1.0, 1.0)


# ---- GPU ---------------------------------------------------------------------------------------

def _check_regions(ctx, picks, levels, what, sources=None):
    fields = _fields(ctx)
    if sources is not None:
        fields = fields[sources[0]:sources[0] + sources[1]]
    reg = ctx.misfit_regions(picks, levels, sources=sources)
    assert_regions_equal(reg, oracle_regions(fields, picks, levels), what)
    assert (reg.npicks == (~np.isnan(picks)).sum(1)).all()
    return fields, reg


@gpu
@pytest.mark.parametrize("kernel", [api.KERNEL_SIMPLE, api.KERNEL_TILED])
@pytest.mark.parametrize("kind", ["random", "hetero", "contrast"])
def test_regions_equal_the_box_restatement(kind, kernel):
    v = make_field(kind, DIMS, 5)
    stations = _stations(6 + 3 * ["random", "hetero", "contrast"].index(kind), seed=1)
    with _context(v, stations, kernel=kernel) as ctx:
        fields = _fields(ctx)
        picks = _events(fields, 24, seed=2)
        picks[3] = np.nan   # no pick at all
        levels = _quantile_levels(fields, picks, seed=3)
        levels[7] = np.nan
        _, reg = _check_regions(ctx, picks, levels, f"{kind} kernel={kernel}")
        assert reg.stats.kernel_launches == 1 and reg.stats.solve_ms > 0
        assert reg.status[3] == api.LOC_NO_PICKS and reg.count[3] == 0 and reg.count[7] == 0
        assert (reg.count[np.isfinite(levels) & (reg.status == api.LOC_OK)] > 0).all()


@gpu
@pytest.mark.parametrize("axis", ["0", "1", "2"])
def test_regions_do_not_depend_on_the_axis_permutation(axis, monkeypatch):
    monkeypatch.setenv("SWEEPTT_WINDOW_AXIS", axis)
    v = make_field("hetero", DIMS, 6)
    with _context(v, _stations(8, seed=3)) as ctx:
        fields = _fields(ctx)
        picks = _events(fields, 16, seed=4)
        _check_regions(ctx, picks, _quantile_levels(fields, picks, seed=5), f"axis {axis}")


@gpu
def test_regions_of_fields_loaded_with_put_tt():
    stations = _stations(7, seed=5)
    with _context(make_field("random", DIMS, 8), stations) as src:
        other = _fields(src)
    with _context(make_field("hetero", DIMS, 9), stations, fields=other) as ctx:
        picks = _events(other, 12, seed=6)
        _check_regions(ctx, picks, _quantile_levels(other, picks, seed=7), "put_tt")


@gpu
def test_levels_at_zero_the_best_misfit_nan_everything_and_signed_zero():
    v = make_field("contrast", DIMS, 13)
    with _context(v, _stations(9, seed=8)) as ctx:
        fields = _fields(ctx)
        rng = np.random.default_rng(9)
        true = rng.integers(int(np.prod(DIMS)), size=20)
        exact = fields.reshape(len(fields), -1)[:, true].T.copy()
        # level 0 with noise-free picks: the true node is inside, and every node inside fits exactly
        _, reg = _check_regions(ctx, exact, np.zeros(20, F), "level 0")
        for e in range(20):
            box = ctx.misfit_box(exact[e])
            c = np.unravel_index(true[e], DIMS)
            assert (reg.lo[e] <= c).all() and (c <= reg.hi[e]).all() and reg.count[e] == (box == 0).sum() >= 1
        # -0.0 is +0
        neg = ctx.misfit_regions(exact, np.full(20, -0.0, F))
        assert_same_regions(neg, reg, "-0.0")
        # the best misfit and its float32 neighbours: the best node goes out below it and comes back in
        picks = _events(fields, 12, seed=10, nan_frac=0)
        loc = ctx.locate_events(picks)
        assert (loc.status == api.LOC_OK).all() and (loc.misfit > 0).all()
        best = loc.misfit
        below = np.nextafter(best, F(0), dtype=F)
        above = np.nextafter(best, F(np.inf), dtype=F)
        r0 = _check_regions(ctx, picks, below, "below the best")[1]
        r1 = _check_regions(ctx, picks, best, "at the best")[1]
        r2 = _check_regions(ctx, picks, above, "above the best")[1]
        assert (r0.count == 0).all() and (r1.count >= 1).all() and (r2.count >= r1.count).all()
        for e in range(12):
            assert (r1.lo[e] <= loc.node[e]).all() and (loc.node[e] <= r1.hi[e]).all()
        assert (r1.origin_min <= loc.origin_time).all() and (loc.origin_time <= r1.origin_max).all()
        # NaN: an empty region, the status still right
        nan = ctx.misfit_regions(picks, np.full(12, np.nan, F))
        assert (nan.count == 0).all() and (nan.status == loc.status).all() and (nan.lo == -1).all()
        assert (nan.moments == 0).all() and np.isnan(nan.origin_min).all() and np.isnan(nan.origin_max).all()
        # above every finite misfit: every node that is neither excluded nor overflowing
        _, every = _check_regions(ctx, picks, np.full(12, FMAX, F), "FLT_MAX")
        for e in range(12):
            assert every.count[e] == np.isfinite(ctx.misfit_box(picks[e])).sum()


@gpu
def test_refused_levels_leave_the_context_as_it_was():
    v = make_field("random", DIMS, 15)
    with _context(v, _stations(6, seed=12)) as ctx:
        fields = _fields(ctx)
        picks = _events(fields, 8, seed=13)
        levels = _quantile_levels(fields, picks, seed=14)
        want = ctx.misfit_regions(picks, levels)
        pool = ctx.pool_bytes
        for bad in (np.inf, -np.inf, -1.0, -FMAX, -np.float32(1e-45)):
            lv = levels.copy()
            lv[5] = bad
            with pytest.raises(P.SweepError, match="level of event 5"):
                ctx.misfit_regions(picks, lv)
            assert ctx.pool_bytes == pool, bad
            assert_same_regions(ctx.misfit_regions(picks, levels), want, f"after level {bad}")
            assert (_bits32(_fields(ctx)) == _bits32(fields)).all()
        lib = P.load_library()
        p, lv = np.ascontiguousarray(picks), np.ascontiguousarray(levels)
        n, st = np.empty(8, np.int64), np.empty(8, np.int32)
        assert not lib.sweeptt_misfit_regions(ctx._h, 0, 6, p.ctypes.data, 8, lv.ctypes.data, None, None, None, None,
                                              st.ctypes.data, None)
        assert b"required" in lib.sweeptt_last_error()
        assert not lib.sweeptt_misfit_regions(ctx._h, 0, 6, p.ctypes.data, 8, None, n.ctypes.data, None, None, None,
                                              st.ctypes.data, None)
        assert b"levels" in lib.sweeptt_last_error()
        # only the required outputs
        assert lib.sweeptt_misfit_regions(ctx._h, 0, 6, p.ctypes.data, 8, lv.ctypes.data, n.ctypes.data, None, None,
                                          None, st.ctypes.data, None)
        assert (n == want.count).all() and (st == want.status).all()
        pk = picks.copy()
        pk[2, 1] = np.inf
        with pytest.raises(P.SweepError, match="INF"):
            ctx.misfit_regions(pk, levels)
        with pytest.raises(P.SweepError, match="not within"):
            ctx.misfit_regions(picks[:, :3], levels, sources=(4, 3))
        assert ctx.pool_bytes == pool
        assert_same_regions(ctx.misfit_regions(picks, levels), want, "after bad arguments")
        assert ctx.misfit_regions(np.zeros((0, 6), F), np.zeros(0, F)).count.shape == (0,)


@gpu
def test_overflowing_misfits_never_enter_and_a_wall_leaves_events_unreached():
    dims = (9, 6, 5)
    v = W.random_field(dims, seed=14)
    v[0, :, :] = np.inf
    v[4, 2, 1] = np.inf
    starts = np.array([(3, 1, 1), (8, 5, 4), (5, 0, 0), (6, 3, 2), (1, 5, 4), (7, 0, 3)], np.int32)
    with _context(v, starts, star="5") as ctx:
        fields = _fields(ctx)
        picks = np.array([[3e38, -3e38, 3e38, -3e38, 1.0, np.nan],
                          [-3e38, np.nan, np.nan, 3e38, np.nan, np.nan],
                          [3e38, 2.0, 5.0, np.nan, 7.0, 1.0],
                          [FMAX, -FMAX, FMAX, -FMAX, FMAX, -FMAX]], F)
        _, reg = _check_regions(ctx, picks, np.full(4, FMAX, F), "overflow")
        assert (reg.status == api.LOC_OK).all() and (reg.count == 0).all()
    star = "5"
    reach = int(np.abs(W.star(star)).max())
    dims = (12 + reach + 1, 9, 10)
    v = W.random_field(dims, seed=12)
    v[6:6 + reach + 1] = np.inf
    stations = np.array([(1, 4, 5), (dims[0] - 2, 4, 5)], np.int32)
    with _context(v, stations, star=star) as ctx:
        picks = np.array([[10, 12], [10, np.nan], [np.nan, 7], [np.nan, np.nan]], F)
        _, reg = _check_regions(ctx, picks, np.full(4, FMAX, F), "wall")
        assert list(reg.status) == [api.LOC_UNREACHED, api.LOC_OK, api.LOC_OK, api.LOC_NO_PICKS]
        assert list(reg.count == 0) == [True, False, False, True]
        nan = ctx.misfit_regions(picks, np.full(4, np.nan, F))
        assert (nan.status == reg.status).all()


@gpu
def test_chunks_repeats_and_source_ranges(monkeypatch):
    v = make_field("hetero", DIMS, 14)
    with _context(v, _stations(10, seed=10)) as ctx:
        fields = _fields(ctx)
        picks = _events(fields, 11, seed=11)
        levels = _quantile_levels(fields, picks, seed=12)
        levels[4] = FMAX   # a large region: many atomics per event
        whole = ctx.misfit_regions(picks, levels)
        assert_same_regions(ctx.misfit_regions(picks, levels), whole, "repeat")
        monkeypatch.setenv("SWEEPTT_LOCATE_CHUNK", "3")
        chunked = ctx.misfit_regions(picks, levels)
        assert chunked.stats.kernel_launches == 4
        assert_same_regions(chunked, whole, "chunks of 3")
        monkeypatch.delenv("SWEEPTT_LOCATE_CHUNK")
        one = _concat([ctx.misfit_regions(picks[e:e + 1], levels[e:e + 1]) for e in range(len(picks))])
        assert_same_regions(one, whole, "one event per call")
        sub = picks[:, 2:7]
        _check_regions(ctx, sub, _quantile_levels(fields[2:7], sub, seed=13), "sources (2, 5)", sources=(2, 5))


@gpu
def test_regions_on_both_sides_of_each_kernel_shape_and_the_station_limit(monkeypatch):
    counts = (225, 226, 452, 453, LOC_MAX_STATIONS)
    rng = np.random.default_rng(31)
    monkeypatch.setenv("SWEEPTT_LOCATE_CHUNK", "37")
    with _station_context(LOC_MAX_STATIONS + 20) as ctx:
        fields = _fields(ctx)
        accepted = []
        for m in range(LOC_MAX_STATIONS - 4, LOC_MAX_STATIONS + 5):
            try:
                ctx.misfit_regions(np.full((1, m), 5, F), np.zeros(1, F), sources=(0, m))
                accepted.append(m)
            except P.SweepError as err:
                assert "shared memory" in str(err)
        largest = max(accepted, default=None)
        assert largest == LOC_MAX_STATIONS, f"largest accepted station count: {largest}"
        assert accepted == list(range(LOC_MAX_STATIONS - 4, largest + 1))
        for m in counts:
            picks = _random_events(fields[:m], 70, rng)
            for e in range(6):   # one pick: every node fits exactly
                picks[e] = np.nan
                picks[e, rng.integers(m)] = F(rng.uniform(0, 50))
            levels = _quantile_levels(fields[:m], picks, seed=m)
            levels[:6] = 0
            _, reg = _check_regions(ctx, picks, levels, f"{m} stations", sources=(0, m))
            assert reg.stats.kernel_launches == 2
            for e in range(6):   # at level 0, every node where the picked station's time is finite
                assert reg.count[e] == np.isfinite(fields[np.nonzero(~np.isnan(picks[e]))[0][0]]).sum()


@gpu
def test_moment_overflow_is_refused_before_any_allocation():
    """n * (n - 1)^2 > 2^63 - 1 first at n = 2^21 + 1 on a line of n nodes: refused there, accepted one node shorter.
    The fields are put, not solved."""
    n = 2 ** 21 + 1
    assert n * (n - 1) ** 2 > 2 ** 63 - 1 >= (n - 1) * (n - 2) ** 2
    for length, ok in ((n - 1, True), (n, False)):
        dims = (length, 1, 1)
        with P.SweepContext(kernel=api.KERNEL_SIMPLE) as ctx:
            ctx.set_model(np.ones(dims, F)); ctx.set_star(W.star("5")); ctx.set_sources([(0, 0, 0)])
            ctx.put_tt(0, np.arange(length, dtype=F).reshape(dims))
            picks = np.array([[5.0]], F)
            ctx.misfit_box(picks[0])   # the context's own buffers, before the region call's
            pool = ctx.pool_bytes
            if ok:
                reg = ctx.misfit_regions(picks, np.zeros(1, F))
                assert reg.count[0] == length and reg.hi[0, 0] == length - 1
            else:
                with pytest.raises(P.SweepError, match="overflow int64"):
                    ctx.misfit_regions(picks, np.zeros(1, F))
                assert ctx.pool_bytes == pool


@gpu
def test_one_shot_location_uncertainty():
    v = make_field("hetero", DIMS, 16)
    stations = _stations(6, seed=14)
    with _context(v, stations) as ctx:
        fields = _fields(ctx)
        picks = _events(fields, 9, seed=15)
        picks[2] = np.nan
        sigma = np.linspace(0.05, 0.5, 9)
        loc, reg = P.location_uncertainty(v, W.star("818"), stations, picks, sigma=sigma, confidence=0.9)
        want_loc = ctx.locate_events(picks)
        assert (loc.node == want_loc.node).all() and (_bits32(loc.misfit) == _bits32(want_loc.misfit)).all()
        levels = P.uncertainty_levels(want_loc, sigma, 0.9)
        assert np.isnan(levels[2]) and np.isfinite(np.delete(levels, 2)).all()
        assert_same_regions(reg, ctx.misfit_regions(picks, levels), "one-shot")
        assert_regions_equal(reg, oracle_regions(fields, picks, levels), "one-shot")
        ok = reg.status == api.LOC_OK
        assert (reg.count[ok] >= 1).all() and np.isfinite(reg.covariance()[ok]).all()


@gpu
def test_full_size_config3_exact_picks():
    """config 3: 111 stations on the 241x241x51 heterogeneous box; 300 events with exact picks: at level 0 every
    region holds the event's true node, and for four events at a wider level the summary equals the box restatement."""
    dims = (241, 241, 51)
    v = W.heterogeneous_field(dims, seed=7)
    stations = W.starts(111)
    with P.SweepContext(kernel=api.KERNEL_TILED) as ctx:
        ctx.set_model(v); ctx.set_star(W.star("818")); ctx.set_sources(stations)
        ctx.run()
        fields = _fields(ctx)
        rng = np.random.default_rng(17)
        true = rng.integers(int(np.prod(dims)), size=300)
        picks = fields.reshape(111, -1)[:, true].T.copy()
        reg = ctx.misfit_regions(picks, np.zeros(300, F))
        assert (reg.status == api.LOC_OK).all() and (reg.count >= 1).all()
        c = np.stack(np.unravel_index(true, dims), 1)
        assert ((reg.lo <= c) & (c <= reg.hi)).all()
        noisy = (picks[:4] + rng.normal(0, 0.05, (4, 111))).astype(F)
        levels = P.uncertainty_levels(ctx.locate_events(noisy), 0.05)
        _check_regions(ctx, noisy, levels, "config 3")
