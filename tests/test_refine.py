"""Sub-node refinement of located events: trilinear station times on a lattice of 1/f of a node in the cube around each
event's centre node (include/sweeptt.h, sweeptt_refine_events / sweeptt_refine_regions; SweepContext.refine_events /
refine_regions, refine_locations).

The yardstick is a numpy restatement of the header's rule (oracle_lattice_times, oracle_refine, oracle_refine_regions):
float64 elementwise operations in the header's order, never fused, with the fields read back with get_tt.  It is itself
checked against scipy's RegularGridInterpolator (a few ulps: its order differs) and, at f = 1, against the node
formula bit for bit.  CPU: the restatement; a C99 client; no fused multiply-add in the new kernels; mean() /
covariance() against Fraction arithmetic; the recentring rule.  GPU (-m gpu): every output bit for bit against the
restatement on random, heterogeneous and contrast models under both kernels, every axis permutation, put_tt, source
ranges, chunking, the cube split and repeats; centres at every corner, edge and face and axes of one node; f = 1, 2, 3,
64; walls, unreachable cubes and events without picks; the station limit; refusals that leave the context as it was;
the properties (f = 1 is the located node, the refined misfit never rises, overlapping cubes agree, f = 1 regions are
the box restricted to the cube, refine_locations' moves lower the key); full-size config 3."""
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
from test_locate import EXCLUDED, _bits32, _bits64, _context, _events, _fields, _stations, oracle_misfit
from test_operator_edges import LOC_MAX_STATIONS, _random_events, _station_context

gpu = pytest.mark.gpu
F = np.float32
FMAX = np.finfo(F).max
DIMS = (21, 18, 16)


# ---- the restatement ---------------------------------------------------------------------------

def _cube(dims, centre, f):
    """The cube's points: u [P, 3] (int64, row-major over the clipped offsets) and their cube-local indices [P]."""
    L = 2 * f + 1
    axes = []
    for a in range(3):
        lo = 0 if centre[a] > 0 else f
        hi = 2 * f if centre[a] < dims[a] - 1 else f
        axes.append(np.arange(lo, hi + 1, dtype=np.int64))
    s = np.stack(np.meshgrid(*axes, indexing="ij"), -1).reshape(-1, 3)
    u = f * (np.asarray(centre, np.int64) - 1) + s
    return u, (s[:, 0] * L + s[:, 1]) * L + s[:, 2]


def oracle_lattice_times(fields, u, f):
    """float64 [S, P]: every station's time at lattice points u [P, 3] by the header's rule."""
    fields = np.asarray(fields, F)
    u = np.asarray(u, np.int64)
    i, r = u // f, u % f
    w = np.array([r_ / f for r_ in range(f)])[r]          # RN(r / f): Python's division is correctly rounded
    step = (r != 0).astype(np.int64)

    def corner(b):
        q = i + step * np.asarray(b)
        return fields[:, q[:, 0], q[:, 1], q[:, 2]].astype(np.float64)

    c = {b: corner(b) for b in np.ndindex(2, 2, 2)}
    inf = np.zeros(c[(0, 0, 0)].shape, bool)
    for v in c.values():
        inf |= v == np.inf

    def lerp(p, q, wa):
        with np.errstate(invalid="ignore"):
            return p + wa * (q - p)

    x = {(b0, b1): lerp(c[(b0, b1, 0)], c[(b0, b1, 1)], w[:, 2]) for b0 in (0, 1) for b1 in (0, 1)}   # axis 2
    y = {b0: lerp(x[(b0, 0)], x[(b0, 1)], w[:, 1]) for b0 in (0, 1)}                                 # axis 1
    t = lerp(y[0], y[1], w[:, 0])                                                                      # axis 0
    return np.where(inf, np.inf, t)


def oracle_point_misfit(times, picks):
    """The node formula over float64 times [S, P]: (misfit f32 [P], t0 [P], k, excluded [P])."""
    picked = [s for s in range(len(picks)) if not np.isnan(picks[s])]
    P_ = times.shape[1]
    excluded = np.zeros(P_, bool)
    for s in picked:
        excluded |= times[s] == np.inf
    acc = np.zeros(P_)
    m = np.zeros(P_)
    with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
        for s in picked:
            acc = acc + (np.float64(picks[s]) - times[s])
        t0 = acc / np.float64(len(picked))
        for s in picked:
            d = (np.float64(picks[s]) - times[s]) - t0
            m = m + d * d
        misfit = m.astype(F)
    misfit[excluded] = np.inf
    return misfit, t0, len(picked), excluded


def _event_cube(fields, picks, centre, f):
    u, local = _cube(fields.shape[1:], centre, f)
    mis, t0, k, excl = oracle_point_misfit(oracle_lattice_times(fields, u, f), picks)
    return u, local, mis, t0, k, excl


def oracle_refine(fields, picks, centres, f):
    """(point int64 [E, 3], misfit f32, origin f64, npicks, status) of every event."""
    E = len(picks)
    point = np.full((E, 3), -1, np.int64)
    misfit = np.full(E, np.inf, F)
    origin = np.full(E, np.nan)
    npicks = np.zeros(E, np.int32)
    status = np.zeros(E, np.int32)
    for e in range(E):
        u, local, mis, t0, k, excl = _event_cube(fields, picks[e], centres[e], f)
        npicks[e] = k
        if k == 0:
            status[e] = api.LOC_NO_PICKS
            continue
        if excl.all():
            status[e] = api.LOC_UNREACHED
            continue
        bits = np.where(excl, EXCLUDED, mis.view(np.uint32).astype(np.uint64))
        j = int(np.argmin((bits << np.uint64(32)) | local.astype(np.uint64)))
        point[e], misfit[e], origin[e] = u[j], mis[j], t0[j]
    return point, misfit, origin, npicks, status


def oracle_refine_regions(fields, picks, centres, f, levels):
    """(count, lo, hi, moments, origin_min, origin_max, status) of R_e = {u in cube : misfit <= levels[e]}."""
    E = len(picks)
    count = np.zeros(E, np.int64)
    lo = np.full((E, 3), -1, np.int64)
    hi = np.full((E, 3), -1, np.int64)
    moments = np.zeros((E, 9), np.int64)
    omin = np.full(E, np.nan)
    omax = np.full(E, np.nan)
    status = np.zeros(E, np.int32)
    for e in range(E):
        u, local, mis, t0, k, excl = _event_cube(fields, picks[e], centres[e], f)
        status[e] = api.LOC_NO_PICKS if k == 0 else api.LOC_UNREACHED if excl.all() else api.LOC_OK
        if k == 0 or np.isnan(levels[e]):
            continue
        R = mis <= F(levels[e])
        count[e] = R.sum()
        if not count[e]:
            continue
        t = u[R] - f * np.asarray(centres[e], np.int64)
        lo[e], hi[e] = u[R].min(0), u[R].max(0)
        moments[e] = [*t.sum(0), *(t * t).sum(0), (t[:, 0] * t[:, 1]).sum(), (t[:, 0] * t[:, 2]).sum(),
                      (t[:, 1] * t[:, 2]).sum()]
        omin[e], omax[e] = t0[R].min(), t0[R].max()
    return count, lo, hi, moments, omin, omax, status


def assert_refined_equal(got, want, what):
    point, misfit, origin, npicks, status = want
    assert (got.status == status).all(), f"{what}: status {got.status} != {status}"
    assert (got.npicks == npicks).all(), what
    bad = np.nonzero((got.point != point).any(1))[0]
    assert not len(bad), f"{what}: points differ for events {bad}: {got.point[bad]} != {point[bad]}"
    assert (_bits32(got.misfit) == _bits32(misfit)).all(), f"{what}: misfit"
    assert (_bits64(got.origin_time) == _bits64(origin)).all(), f"{what}: origin time"


def assert_refined_regions_equal(got, want, what):
    count, lo, hi, moments, omin, omax, status = want
    assert (got.status == status).all(), f"{what}: status {got.status} != {status}"
    bad = np.nonzero(got.count != count)[0]
    assert not len(bad), f"{what}: counts differ for events {bad}: {got.count[bad]} != {count[bad]}"
    assert (got.lo == lo).all() and (got.hi == hi).all(), f"{what}: bounding box"
    assert (got.moments == moments).all(), f"{what}: moments"
    assert (_bits64(got.origin_min) == _bits64(omin)).all(), f"{what}: origin min"
    assert (_bits64(got.origin_max) == _bits64(omax)).all(), f"{what}: origin max"


def _same_refined(a, b, what):
    for f in ("point", "npicks", "status"):
        assert (getattr(a, f) == getattr(b, f)).all(), f"{what}: {f}"
    assert (_bits32(a.misfit) == _bits32(b.misfit)).all() and (_bits64(a.origin_time) == _bits64(b.origin_time)).all()


def _same_regions(a, b, what):
    for f in ("count", "lo", "hi", "moments", "npicks", "status"):
        assert (getattr(a, f) == getattr(b, f)).all(), f"{what}: {f}"
    for f in ("origin_min", "origin_max"):
        assert (_bits64(getattr(a, f)) == _bits64(getattr(b, f))).all(), f"{what}: {f}"


def _cube_levels(fields, picks, centres, f, seed):
    """A level per event between its best cube misfit and well above it."""
    rng = np.random.default_rng(seed)
    levels = np.empty(len(picks), F)
    for e in range(len(picks)):
        mis = _event_cube(fields, picks[e], centres[e], f)[2]
        fin = mis[np.isfinite(mis)]
        levels[e] = F(np.quantile(fin, rng.choice([0.0, 0.01, 0.1, 0.5]))) if len(fin) else F(1)
    return levels


# ---- CPU ---------------------------------------------------------------------------------------

def test_restatement_agrees_with_scipy_and_is_the_node_formula_on_nodes():
    from scipy.interpolate import RegularGridInterpolator
    rng = np.random.default_rng(1)
    dims = (6, 5, 4)
    fields = rng.uniform(0, 60, (3, *dims)).astype(F)
    for f in (1, 2, 3, 7):
        u = np.stack([rng.integers(0, f * (n - 1) + 1, 300) for n in dims], 1)
        got = oracle_lattice_times(fields, u, f)
        for s in range(3):
            rgi = RegularGridInterpolator([np.arange(n) for n in dims], fields[s].astype(np.float64), method="linear")
            want = rgi(u / f)
            assert np.all(np.abs(got[s] - want) <= 8 * np.spacing(np.maximum(np.abs(want), 1.0))), f
        on = (u % f == 0).all(1)
        q = u[on] // f
        assert (got[:, on] == fields[:, q[:, 0], q[:, 1], q[:, 2]]).all()   # nodes: exactly their time
    # f = 1: the cube misfits are the node formula's, bit for bit
    picks = (fields[:, 2, 3, 1] + F(4) + rng.normal(0, 0.1, 3)).astype(F)
    mis_box = oracle_misfit(fields, picks)[0]
    u, _, mis, *_ = _event_cube(fields, picks, (2, 3, 1), 1)
    assert (_bits32(mis) == _bits32(mis_box[u[:, 0], u[:, 1], u[:, 2]])).all()
    # an infinite corner gives +inf wherever it is read, and only there
    fields[1, 3, 2, 2] = np.inf
    t = oracle_lattice_times(fields, np.array([[6, 4, 4], [5, 4, 4], [7, 4, 4], [6, 3, 4], [4, 4, 4]]), 2)
    assert (t[1, :4] == np.inf).all() and np.isfinite(t[1, 4]) and np.isfinite(t[[0, 2]]).all()


def test_recentring_keeps_the_best_point_in_the_new_cube():
    for f in (1, 2, 3, 8, 64):
        for n in (1, 2, 5):
            for u in range(f * (n - 1) + 1):
                ref = api.RefinedLocations(np.array([[u, 0, 0]]), f, np.zeros((1, 3), np.int32), np.zeros(1, F),
                                           np.zeros(1), np.ones(1, np.int32), np.zeros(1, np.int32), None, (n, 1, 1))
                c = int(P.recentre(ref)[0, 0])
                assert 0 <= c < n and 2 * abs(u - f * c) <= f, (f, n, u, c)


def test_on_edge_and_truncated_are_interior_faces_only():
    f, dims = 4, (5, 1, 3)
    centre = np.array([[2, 0, 0]] * 4 + [[3, 0, 1]], np.int32)
    point = np.array([[12, 0, 0], [10, 0, 4], [8, 0, 0], [9, 0, 3], [16, 0, 8]])
    status = np.array([0, 0, 0, 0, 0], np.int32)
    ref = api.RefinedLocations(point, f, centre, np.zeros(5, F), np.zeros(5), np.ones(5, np.int32), status, None, dims)
    # [12,0,0]: t0 = +f, interior; [10,0,4]: t2 = +f at u2 = 4 < 8, interior; [8,0,0]: the centre; [9,0,3]: inside
    # the cube; [16,0,8]: t0 = t2 = +f, but on the box's faces
    assert list(ref.on_edge) == [True, True, False, False, False]
    ref.status[0] = api.LOC_UNREACHED
    assert not ref.on_edge[0]
    reg = api.RefinedRegions(np.array([3, 1, 0]), np.array([[4, 0, 0], [8, 0, 0], [-1, -1, -1]]),
                             np.array([[9, 0, 2], [8, 0, 0], [-1, -1, -1]]), np.zeros((3, 9), np.int64),
                             np.zeros(3), np.zeros(3), np.array([[2, 0, 0], [2, 0, 0], [2, 0, 0]], np.int32), f,
                             np.ones(3, np.int32), np.zeros(3, np.int32), None, dims)
    assert list(reg.truncated) == [True, False, False]


@pytest.mark.skipif(shutil.which("cuobjdump") is None, reason="cuobjdump not on PATH")
def test_refine_kernels_never_fuse_multiply_add():
    out = subprocess.run(["cuobjdump", "-sass", str(P.lib_path())], capture_output=True, text=True, check=True).stdout
    funcs, name = {}, None
    for line in out.splitlines():
        mm = re.search(r"Function : (\S+)", line)
        if mm:
            name = mm.group(1)
            funcs[name] = []
        elif name and re.match(r"\s+/\*[0-9a-f]{4,6}\*/", line):
            funcs[name].append(line)
    kernels = {k: v for k, v in funcs.items() if "refine" in k}
    assert len(kernels) == 3, sorted(kernels)   # refine_kernel, refine_regions_kernel, refine_finish_kernel
    for k, lines in kernels.items():
        text = "\n".join(lines)
        assert "DADD" in text and "DMUL" in text, k
        assert not re.search(r"\b[DF]FMA2?\b", text), f"{k}: fused multiply-add found"


def test_c99_client_calls_both_refine_entry_points(tmp_path):
    """A strict C99 client compiles and links.  Without a GPU each call fails with "null context"; with one, a 4x4x4
    box and one station: one pick fits every point exactly, so the best point is the cube's first and level 0 takes
    the whole cube."""
    src = tmp_path / "client.c"
    src.write_text(r'''
#include <stdio.h>
#include "sweeptt.h"
int main(void) {
  struct FS fs[7] = {{1, 0, 0, 0.f}, {-1, 0, 0, 0.f}, {0, 1, 0, 0.f}, {0, -1, 0, 0.f}, {0, 0, 1, 0.f},
                     {0, 0, -1, 0.f}, {1, 1, 1, 0.f}};
  struct START st[1] = {{0, 0, 0}}, centre[1] = {{1, 2, 3}};
  float v[64], picks[1] = {30.f}, misfit[1], levels[1] = {0.f};
  int64_t point[3], count[1], bbox[6], moments[9];
  double origin[1], range[2];
  int32_t npicks[1], status[1];
  int i;
  sweeptt_stats stats;
  sweeptt_ctx *ctx;
  for (i = 0; i < 64; i++) v[i] = 1.f;
  sweeptt_star_fill_distances(fs, 7, 10.0f);
  ctx = sweeptt_create(NULL);
  if (!ctx) {
    if (sweeptt_refine_events(NULL, 0, 1, picks, 1, centre, 4, point, misfit, origin, npicks, status, &stats)) return 2;
    printf("%s\n", sweeptt_last_error());
    if (sweeptt_refine_regions(NULL, 0, 1, picks, 1, centre, 4, levels, count, bbox, moments, range, status, &stats))
      return 2;
    printf("%s\n", sweeptt_last_error());
    return 0;
  }
  if (!sweeptt_set_model(ctx, v, 4, 4, 4) || !sweeptt_set_star(ctx, fs, 7) || !sweeptt_set_sources(ctx, st, 1) ||
      !sweeptt_run(ctx, NULL) ||
      !sweeptt_refine_events(ctx, 0, 1, picks, 1, centre, 4, point, misfit, origin, npicks, status, &stats) ||
      !sweeptt_refine_regions(ctx, 0, 1, picks, 1, centre, 4, levels, count, bbox, moments, range, status, &stats)) {
    printf("%s\n", sweeptt_last_error());
    return 3;
  }
  sweeptt_destroy(ctx);
  if (status[0] != SWEEPTT_LOC_OK || npicks[0] != 1 || point[0] != 0 || point[1] != 4 || point[2] != 8) return 4;
  if (misfit[0] != 0.f || count[0] != 9 * 9 * 5 || bbox[0] != 0 || bbox[3] != 8 || bbox[5] != 12) return 5;
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
        assert r.stdout.count("null context") == 2, r.stdout


def test_refined_mean_and_covariance_are_the_exact_quotients_rounded_once():
    rng = np.random.default_rng(41)
    f = 7
    centre = np.array([[3, 9, 2], [0, 0, 0], [100, 5, 7], [1, 1, 1]], np.int32)
    sets = [rng.integers(-f, f + 1, (n, 3)) for n in (1, 2, 500)] + [np.zeros((0, 3), np.int64)]
    moments = np.zeros((4, 9), np.int64)
    for e, t in enumerate(sets):
        t = t.astype(np.int64)
        moments[e] = [*t.sum(0), *(t * t).sum(0), (t[:, 0] * t[:, 1]).sum(), (t[:, 0] * t[:, 2]).sum(),
                      (t[:, 1] * t[:, 2]).sum()]
    count = np.array([len(t) for t in sets], np.int64)
    z = np.zeros((4, 3), np.int64)
    reg = api.RefinedRegions(count, z, z, moments, np.zeros(4), np.zeros(4), centre, f, np.ones(4, np.int32),
                             np.zeros(4, np.int32))
    mean, cov = reg.mean(), reg.covariance()
    for e, t in enumerate(sets[:3]):
        n = len(t)
        pos = [[Fraction(int(centre[e, a])) + Fraction(int(x[a]), f) for a in range(3)] for x in t]
        for a in range(3):
            ma = sum(p[a] for p in pos) / n
            assert mean[e, a] == float(ma)
            for b in range(3):
                mb = sum(p[b] for p in pos) / n
                assert cov[e, a, b] == float(sum((p[a] - ma) * (p[b] - mb) for p in pos) / n), (e, a, b)
    assert (cov[0] == 0).all() and np.isnan(mean[3]).all() and np.isnan(cov[3]).all()


# ---- GPU ---------------------------------------------------------------------------------------

def _check_refine(ctx, picks, centres, f, what, sources=None, levels=None):
    fields = _fields(ctx)
    if sources is not None:
        fields = fields[sources[0]:sources[0] + sources[1]]
    ref = ctx.refine_events(picks, centres, f, sources=sources)
    assert_refined_equal(ref, oracle_refine(fields, picks, centres, f), what)
    assert ref.stats.solve_ms > 0
    if levels is None:
        levels = _cube_levels(fields, picks, centres, f, seed=f)
    reg = ctx.refine_regions(picks, centres, f, levels, sources=sources)
    assert_refined_regions_equal(reg, oracle_refine_regions(fields, picks, centres, f, levels), what)
    assert (reg.npicks == (~np.isnan(picks)).sum(1)).all()
    return fields, ref, reg


def _random_centres(n, dims, seed):
    return np.stack([np.random.default_rng(seed).integers(0, d, n) for d in dims], 1).astype(np.int32)


@gpu
@pytest.mark.parametrize("kernel", [api.KERNEL_SIMPLE, api.KERNEL_TILED])
@pytest.mark.parametrize("kind", ["random", "hetero", "contrast"])
def test_refinement_equals_the_restatement(kind, kernel):
    v = make_field(kind, DIMS, 21)
    with _context(v, _stations(7, seed=4), kernel=kernel) as ctx:
        fields = _fields(ctx)
        picks = _events(fields, 12, seed=5)
        picks[2] = np.nan
        loc = ctx.locate_events(picks)
        centres = np.where(loc.status[:, None] == api.LOC_OK, loc.node, 3).astype(np.int32)
        centres[5:8] = _random_centres(3, DIMS, 6)
        _, ref, reg = _check_refine(ctx, picks, centres, 3, f"{kind} kernel={kernel}")
        assert ref.stats.kernel_launches == 2 and reg.stats.kernel_launches == 1
        assert ref.status[2] == api.LOC_NO_PICKS and (ref.point[2] == -1).all() and reg.count[2] == 0


@gpu
@pytest.mark.parametrize("axis", ["0", "1", "2"])
def test_refinement_does_not_depend_on_the_axis_permutation(axis, monkeypatch):
    monkeypatch.setenv("SWEEPTT_WINDOW_AXIS", axis)
    with _context(make_field("hetero", DIMS, 22), _stations(6, seed=7)) as ctx:
        fields = _fields(ctx)
        picks = _events(fields, 8, seed=8)
        _check_refine(ctx, picks, _random_centres(8, DIMS, 9), 4, f"axis {axis}")


@gpu
def test_refinement_of_fields_loaded_with_put_tt():
    stations = _stations(5, seed=10)
    with _context(make_field("random", DIMS, 23), stations) as src:
        other = _fields(src)
    with _context(make_field("hetero", DIMS, 24), stations, fields=other) as ctx:
        picks = _events(other, 6, seed=11)
        _check_refine(ctx, picks, _random_centres(6, DIMS, 12), 2, "put_tt")


@gpu
def test_chunks_cube_splits_repeats_and_source_ranges(monkeypatch):
    with _context(make_field("hetero", DIMS, 25), _stations(9, seed=13)) as ctx:
        fields = _fields(ctx)
        picks = _events(fields, 7, seed=14)
        centres = _random_centres(7, DIMS, 15)
        levels = _cube_levels(fields, picks, centres, 3, seed=16)
        levels[3] = FMAX
        ref = ctx.refine_events(picks, centres, 3)
        reg = ctx.refine_regions(picks, centres, 3, levels)
        _same_refined(ctx.refine_events(picks, centres, 3), ref, "repeat")
        _same_regions(ctx.refine_regions(picks, centres, 3, levels), reg, "repeat")
        for chunk, points in (("1", None), ("3", "1"), (None, "37"), (None, "100000")):
            for var, val in (("SWEEPTT_LOCATE_CHUNK", chunk), ("SWEEPTT_REFINE_POINTS", points)):
                if val is None:
                    monkeypatch.delenv(var, raising=False)
                else:
                    monkeypatch.setenv(var, val)
            got = ctx.refine_events(picks, centres, 3)
            _same_refined(got, ref, f"chunk {chunk}, points {points}")
            _same_regions(ctx.refine_regions(picks, centres, 3, levels), reg, f"chunk {chunk}, points {points}")
            if chunk == "1":
                assert got.stats.kernel_launches == 8
        monkeypatch.delenv("SWEEPTT_LOCATE_CHUNK", raising=False)
        monkeypatch.delenv("SWEEPTT_REFINE_POINTS", raising=False)
        sub = picks[:, 2:6]
        _check_refine(ctx, sub, centres, 3, "sources (2, 4)", sources=(2, 4))


@gpu
def test_centres_at_every_corner_edge_and_face_and_axes_of_one_node():
    with _context(make_field("random", DIMS, 26), _stations(5, seed=17)) as ctx:
        fields = _fields(ctx)
        where = [(0, d // 2, d - 1) for d in DIMS]
        centres = np.array([(a, b, c) for a in where[0] for b in where[1] for c in where[2]], np.int32)
        picks = _events(fields, len(centres), seed=18)
        for f in (1, 2, 3):
            _check_refine(ctx, picks, centres, f, f"27 positions, f = {f}")
    rng = np.random.default_rng(19)
    for dims in ((1, 9, 7), (8, 1, 1), (1, 1, 1)):   # fields put, not solved
        stations = np.array([(0, 0, 0), tuple(d - 1 for d in dims), tuple(d // 2 for d in dims)], np.int32)
        put = rng.uniform(0, 40, (3, *dims)).astype(F)
        with _context(np.ones(dims, F), stations, star="5", fields=put) as ctx:
            fields = _fields(ctx)
            assert (fields == put).all()
            picks = _random_events(fields, 6, rng, nan_frac=0.2)
            centres = _random_centres(6, dims, 20)
            _check_refine(ctx, picks, centres, 5, f"dims {dims}")


@gpu
def test_subdiv_64_and_the_largest_cube():
    with _context(make_field("hetero", DIMS, 27), _stations(4, seed=21)) as ctx:
        fields = _fields(ctx)
        picks = _events(fields, 2, seed=22, nan_frac=0)
        centres = np.array([(10, 9, 8), (0, 17, 7)], np.int32)
        _, ref, reg = _check_refine(ctx, picks, centres, 64, "f = 64")
        assert (ref.status == api.LOC_OK).all()
        full = ctx.refine_regions(picks, centres, 64, np.full(2, FMAX, F))
        assert full.count[0] == 129 ** 3 and full.count[1] == 65 * 65 * 129


@gpu
def test_a_wall_excludes_points_and_leaves_cubes_unreached():
    star = "5"
    reach = int(np.abs(W.star(star)).max())
    dims = (12 + reach + 1, 9, 10)
    v = W.random_field(dims, seed=12)
    v[6:6 + reach + 1] = np.inf
    stations = np.array([(1, 4, 5), (dims[0] - 2, 4, 5)], np.int32)
    with _context(v, stations, star=star) as ctx:
        fields = _fields(ctx)
        picks = np.array([[10, 12], [10, np.nan], [np.nan, 7], [np.nan, np.nan], [10, 12], [10, np.nan]], F)
        centres = np.array([(3, 4, 5), (5, 4, 5), (6 + reach + 1, 4, 5), (3, 4, 5), (6, 4, 5), (6 + reach, 2, 2)],
                           np.int32)
        _, ref, reg = _check_refine(ctx, picks, centres, 4, "wall", levels=np.full(6, FMAX, F))
        assert list(ref.status) == [api.LOC_UNREACHED, api.LOC_OK, api.LOC_OK, api.LOC_NO_PICKS, api.LOC_UNREACHED,
                                    api.LOC_UNREACHED]
        # centre (5, 4, 5) sits next to the wall: its cube's points that read the wall are excluded
        mis = _event_cube(fields, picks[1], centres[1], 4)[2]
        assert np.isinf(mis).any() and np.isfinite(mis).any()


@gpu
def test_refusals_leave_the_context_as_it_was():
    with _context(make_field("random", DIMS, 28), _stations(6, seed=23)) as ctx:
        fields = _fields(ctx)
        picks = _events(fields, 5, seed=24)
        centres = _random_centres(5, DIMS, 25)
        levels = _cube_levels(fields, picks, centres, 3, seed=26)
        want = ctx.refine_events(picks, centres, 3)
        want_reg = ctx.refine_regions(picks, centres, 3, levels)
        want_loc = ctx.locate_events(picks)
        pool = ctx.pool_bytes

        def unchanged(what):
            assert ctx.pool_bytes == pool, what
            _same_refined(ctx.refine_events(picks, centres, 3), want, what)
            _same_regions(ctx.refine_regions(picks, centres, 3, levels), want_reg, what)
            loc = ctx.locate_events(picks)
            assert (loc.node == want_loc.node).all() and (_bits32(loc.misfit) == _bits32(want_loc.misfit)).all()

        for a, bad in ((0, -1), (0, DIMS[0]), (1, DIMS[1]), (2, -5), (2, DIMS[2])):
            c = centres.copy()
            c[3, a] = bad
            with pytest.raises(P.SweepError, match="centre of event 3"):
                ctx.refine_events(picks, c, 3)
            with pytest.raises(P.SweepError, match="centre of event 3"):
                ctx.refine_regions(picks, c, 3, levels)
            unchanged(f"centre {c[3]}")
        for f in (0, 65, -1):
            with pytest.raises(P.SweepError, match="subdiv"):
                ctx.refine_events(picks, centres, f)
            with pytest.raises(P.SweepError, match="subdiv"):
                ctx.refine_regions(picks, centres, f, levels)
            unchanged(f"subdiv {f}")
        for bad in (np.inf, -np.inf, -1.0, -np.float32(1e-45)):
            lv = levels.copy()
            lv[4] = bad
            with pytest.raises(P.SweepError, match="level of event 4"):
                ctx.refine_regions(picks, centres, 3, lv)
            unchanged(f"level {bad}")
        _same_regions(ctx.refine_regions(picks, centres, 3, np.full(5, -0.0, F)),
                      ctx.refine_regions(picks, centres, 3, np.zeros(5, F)), "-0.0")
        lib = P.load_library()
        p, lv = np.ascontiguousarray(picks), np.ascontiguousarray(levels)
        pt, n, st = np.empty((5, 3), np.int64), np.empty(5, np.int64), np.empty(5, np.int32)
        assert not lib.sweeptt_refine_events(ctx._h, 0, 6, p.ctypes.data, 5, None, 3, pt.ctypes.data, None, None, None,
                                             st.ctypes.data, None)
        assert b"null centres" in lib.sweeptt_last_error()
        assert not lib.sweeptt_refine_regions(ctx._h, 0, 6, p.ctypes.data, 5, None, 3, lv.ctypes.data, n.ctypes.data,
                                              None, None, None, st.ctypes.data, None)
        assert b"null centres" in lib.sweeptt_last_error()
        c = np.ascontiguousarray(centres)
        assert not lib.sweeptt_refine_events(ctx._h, 0, 6, p.ctypes.data, 5, c.ctypes.data, 3, None, None, None, None,
                                             st.ctypes.data, None)
        assert b"required" in lib.sweeptt_last_error()
        assert not lib.sweeptt_refine_regions(ctx._h, 0, 6, p.ctypes.data, 5, c.ctypes.data, 3, None, n.ctypes.data,
                                              None, None, None, st.ctypes.data, None)
        assert b"levels" in lib.sweeptt_last_error()
        # only the required outputs
        assert lib.sweeptt_refine_events(ctx._h, 0, 6, p.ctypes.data, 5, c.ctypes.data, 3, pt.ctypes.data, None, None,
                                         None, st.ctypes.data, None)
        assert (pt == want.point).all() and (st == want.status).all()
        pk = picks.copy()
        pk[1, 2] = -np.inf
        with pytest.raises(P.SweepError, match="INF"):
            ctx.refine_events(pk, centres, 3)
        with pytest.raises(P.SweepError, match="not within"):
            ctx.refine_events(picks[:, :3], centres, 3, sources=(4, 3))
        unchanged("bad arguments")
        assert ctx.refine_events(np.zeros((0, 6), F), np.zeros((0, 3), np.int32), 3).point.shape == (0, 3)
        assert ctx.refine_regions(np.zeros((0, 6), F), np.zeros((0, 3), np.int32), 3, np.zeros(0, F)).count.shape == (0,)


@gpu
def test_station_limit_of_the_location_calls(monkeypatch):
    rng = np.random.default_rng(32)
    monkeypatch.setenv("SWEEPTT_LOCATE_CHUNK", "29")
    with _station_context(LOC_MAX_STATIONS + 1) as ctx:
        fields = _fields(ctx)
        dims = fields.shape[1:]
        for m in (225, 226, 452, 453, LOC_MAX_STATIONS):
            picks = _random_events(fields[:m], 40, rng)
            centres = _random_centres(40, dims, m)
            _check_refine(ctx, picks, centres, 2, f"{m} stations", sources=(0, m))
        m = LOC_MAX_STATIONS + 1
        pool = ctx.pool_bytes
        with pytest.raises(P.SweepError, match="shared memory"):
            ctx.refine_events(np.full((1, m), 5, F), np.zeros((1, 3), np.int32), 2, sources=(0, m))
        with pytest.raises(P.SweepError, match="shared memory"):
            ctx.refine_regions(np.full((1, m), 5, F), np.zeros((1, 3), np.int32), 2, np.zeros(1, F), sources=(0, m))
        assert ctx.pool_bytes == pool


@gpu
def test_properties_against_the_grid_search():
    """f = 1 at the located node is that node, bit for bit; the refined misfit never rises; overlapping cubes give
    the same misfit at the same point; f = 1 regions are the misfit box under the level inside the 27-node cube."""
    with _context(make_field("hetero", DIMS, 29), _stations(8, seed=27)) as ctx:
        fields = _fields(ctx)
        picks = _events(fields, 16, seed=28)
        picks[4] = np.nan
        loc = ctx.locate_events(picks)
        ok = loc.status == api.LOC_OK
        centres = np.where(ok[:, None], loc.node, 0).astype(np.int32)
        one = ctx.refine_events(picks, centres, 1)
        assert (one.status == loc.status).all()
        assert (one.point[ok] == loc.node[ok]).all()
        assert (_bits32(one.misfit) == _bits32(loc.misfit)).all()
        assert (_bits64(one.origin_time[ok]) == _bits64(loc.origin_time[ok])).all()
        for f in (2, 3, 5, 8):
            ref = ctx.refine_events(picks, centres, f)
            assert (ref.misfit[ok] <= loc.misfit[ok]).all(), f
            # the best point again, in the cube around the node nearest it: its misfit is the same, so the new best
            # is no worse, and a region at that misfit holds it
            moved = ctx.refine_events(picks, P.recentre(ref), f)
            assert (moved.misfit[ok] <= ref.misfit[ok]).all()
            same = ok & (moved.point == ref.point).all(1)
            assert (_bits32(moved.misfit[same]) == _bits32(ref.misfit[same])).all()
            assert (_bits64(moved.origin_time[same]) == _bits64(ref.origin_time[same])).all()
            reg = ctx.refine_regions(picks, P.recentre(ref), f, np.where(ok, ref.misfit, np.nan).astype(F))
            assert (reg.count[ok] >= 1).all()
            assert ((reg.lo[ok] <= ref.point[ok]) & (ref.point[ok] <= reg.hi[ok])).all()
        levels = _cube_levels(fields, picks, centres, 1, seed=30)
        reg = ctx.refine_regions(picks, centres, 1, levels)
        for e in np.nonzero(ok)[0]:
            box = ctx.misfit_box(picks[e])
            u, _ = _cube(DIMS, centres[e], 1)
            inside = u[box[u[:, 0], u[:, 1], u[:, 2]] <= levels[e]]
            assert reg.count[e] == len(inside)
            if len(inside):
                assert (reg.lo[e] == inside.min(0)).all() and (reg.hi[e] == inside.max(0)).all()


@gpu
def test_refine_locations_moves_lower_the_key_and_stop():
    v = make_field("hetero", DIMS, 30)
    stations = _stations(7, seed=31)
    with _context(v, stations) as ctx:
        fields = _fields(ctx)
        picks = _events(fields, 10, seed=32)
        picks[6] = np.nan
        for f, max_moves in ((2, 0), (4, 1), (4, 8)):
            loc, ref = P.refine_locations(v, W.star("818"), stations, picks, subdiv=f, max_moves=max_moves)
            want_loc = ctx.locate_events(picks)
            assert (loc.node == want_loc.node).all() and (loc.status == want_loc.status).all()
            ok = loc.status == api.LOC_OK
            # the same loop by hand, checking each move against the restatement and the key order
            cur = ctx.refine_events(picks[ok], loc.node[ok], f)
            moves = np.zeros(ok.sum(), np.int32)
            for _ in range(max_moves):
                edge = np.nonzero(cur.on_edge)[0]
                if not len(edge):
                    break
                nxt = ctx.refine_events(picks[ok][edge], P.recentre(cur)[edge], f)
                assert_refined_equal(nxt, oracle_refine(fields, picks[ok][edge], P.recentre(cur)[edge], f), "move")
                old = [(int(_bits32(cur.misfit[e])), tuple(cur.point[e])) for e in edge]
                cur.point[edge], cur.centre[edge], cur.misfit[edge] = nxt.point, nxt.centre, nxt.misfit
                cur.origin_time[edge] = nxt.origin_time
                moves[edge] += 1
                still = cur.on_edge
                for j, e in enumerate(edge):   # a lower key, or the same point, now off the cube's faces
                    new = (int(_bits32(cur.misfit[e])), tuple(cur.point[e]))
                    assert new < old[j] or (new == old[j] and not still[e]), (e, old[j], new)
            assert (ref.point[ok] == cur.point).all() and (_bits32(ref.misfit[ok]) == _bits32(cur.misfit)).all()
            assert (ref.moves[ok] == moves).all() and ref.moves.max() <= max_moves
            assert (ref.misfit[ok] <= loc.misfit[ok]).all()
            assert (ref.point[~ok] == -1).all() and np.isnan(ref.position[~ok]).all()
            assert np.allclose(ref.position[ok], ref.point[ok] / f)
        loc, ref, reg = P.refine_locations(v, W.star("818"), stations, picks, subdiv=3, sigma=0.05)
        levels = P.uncertainty_levels(ref, 0.05)
        assert np.isnan(levels[6]) and reg.count[6] == 0
        assert_refined_regions_equal(reg, oracle_refine_regions(fields, picks, ref.centre, 3, levels), "one-shot")
        ok = reg.status == api.LOC_OK
        assert (reg.count[ok] >= 1).all() and np.isfinite(reg.mean()[ok]).all()


@gpu
def test_full_size_config3_sample():
    """config 3: 111 stations on the 241x241x51 heterogeneous box, located events refined at f = 4: the kernel
    against the restatement on a sample of events (picks as tools/locate_bench.py makes them)."""
    import sys
    sys.path.insert(0, str(ROOT / "tools"))
    from locate_bench import make_picks
    dims = (241, 241, 51)
    with P.SweepContext(kernel=api.KERNEL_TILED) as ctx:
        ctx.set_model(W.heterogeneous_field(dims, seed=7)); ctx.set_star(W.star("818")); ctx.set_sources(W.starts(111))
        ctx.run()
        picks = make_picks(ctx, 200, 200)
        loc = ctx.locate_events(picks)
        ok = loc.status == api.LOC_OK
        centres = np.where(ok[:, None], loc.node, 0).astype(np.int32)
        ref = ctx.refine_events(picks, centres, 4)
        assert (ref.misfit[ok] <= loc.misfit[ok]).all()
        levels = P.uncertainty_levels(ref, 0.05)
        reg = ctx.refine_regions(picks, centres, 4, levels)
        sample = np.random.default_rng(3).choice(len(picks), 6, replace=False)
        fields = np.stack([ctx.get_tt(s) for s in range(111)])
        for e in sample:
            want = oracle_refine(fields, picks[e:e + 1], centres[e:e + 1], 4)
            assert_refined_equal(api.RefinedLocations(ref.point[e:e + 1], 4, centres[e:e + 1], ref.misfit[e:e + 1],
                                                      ref.origin_time[e:e + 1], ref.npicks[e:e + 1],
                                                      ref.status[e:e + 1], None), want, f"config 3 event {e}")
            want = oracle_refine_regions(fields, picks[e:e + 1], centres[e:e + 1], 4, levels[e:e + 1])
            got = api.RefinedRegions(*(x[e:e + 1] for x in (reg.count, reg.lo, reg.hi, reg.moments, reg.origin_min,
                                                            reg.origin_max, reg.centre)), 4, reg.npicks[e:e + 1],
                                     reg.status[e:e + 1])
            assert_refined_regions_equal(got, want, f"config 3 event {e}")
