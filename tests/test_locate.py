"""Event location by grid search over the stations' travel-time fields (include/sweeptt.h, sweeptt_locate_events /
sweeptt_misfit_box).

The yardstick is a numpy restatement of the header's formula (oracle_misfit): float64 elementwise operations, the
stations in increasing order, never np.sum (which sums pairwise).  CPU: the oracle against a plain float64 least-squares
fit; the new kernels never fuse a multiply-add; a C99 client links against both entry points.  GPU (-m gpu), with the
fields read back with get_tt so the oracle sees exactly what the device used: misfit boxes bit for bit on random,
heterogeneous and contrast models under both kernels, every axis permutation and put_tt; every event's node, misfit,
origin time, pick count and status bit for bit; ties; NaN picks; unreachable events; noise-free picks; chunking,
determinism, source ranges; refusals that leave the context as it was; full-size config 3."""
import re
import shutil
import subprocess

import numpy as np
import pytest
import torch

import uoparallel_seismic_project_b200 as P
from uoparallel_seismic_project_b200 import api, workloads as W

from conftest import ROOT, make_field

gpu = pytest.mark.gpu
F = np.float32
EXCLUDED = np.uint64(0x7F800001)   # key bits of an excluded node (ranks after every float32 misfit, +inf included)


# ---- the oracle --------------------------------------------------------------------------------

def oracle_misfit(fields, picks):
    """The header's formula at every node.  fields [S, ...] float32, picks [S] float32 (NaN = no pick).
    Returns (misfit float32 [...] with +inf where excluded, t0 float64 [...], k, excluded bool [...])."""
    fields = np.asarray(fields, F)
    picked = [s for s in range(len(picks)) if not np.isnan(picks[s])]
    shape = fields.shape[1:]
    excluded = np.zeros(shape, bool)
    for s in picked:
        excluded |= fields[s] == np.inf
    acc = np.zeros(shape)
    m = np.zeros(shape)
    with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
        for s in picked:
            acc = acc + (np.float64(picks[s]) - fields[s].astype(np.float64))
        t0 = acc / np.float64(len(picked))
        for s in picked:
            u = (np.float64(picks[s]) - fields[s].astype(np.float64)) - t0
            m = m + u * u
        misfit = m.astype(F)
    misfit[excluded] = np.inf
    return misfit, t0, len(picked), excluded


def oracle_locate(fields, picks):
    """Every event of picks [E, S]: (node int32 [E, 3], misfit f32 [E], origin f64 [E], npicks [E], status [E])."""
    dims = np.asarray(fields).shape[1:]
    E = len(picks)
    node = np.full((E, 3), -1, np.int32)
    misfit = np.full(E, np.inf, F)
    origin = np.full(E, np.nan)
    npicks = np.zeros(E, np.int32)
    status = np.zeros(E, np.int32)
    index = np.arange(int(np.prod(dims)), dtype=np.uint64)
    for e, p in enumerate(picks):
        mis, t0, k, excl = oracle_misfit(fields, p)
        npicks[e] = k
        if k == 0:
            status[e] = api.LOC_NO_PICKS
            continue
        if excl.all():
            status[e] = api.LOC_UNREACHED
            continue
        bits = np.where(excl, EXCLUDED, mis.view(np.uint32).astype(np.uint64)).ravel()
        j = int(np.argmin((bits << np.uint64(32)) | index))
        node[e] = np.unravel_index(j, dims)
        misfit[e], origin[e] = mis.ravel()[j], t0.ravel()[j]
    return node, misfit, origin, npicks, status


def _bits32(a):
    return np.ascontiguousarray(a, F).view(np.uint32)


def _bits64(a):
    return np.ascontiguousarray(a, np.float64).view(np.uint64)


def assert_locations_equal(got, want, what):
    node, misfit, origin, npicks, status = want
    assert (got.status == status).all(), f"{what}: status {got.status} != {status}"
    assert (got.npicks == npicks).all(), what
    assert (got.node == node).all(), f"{what}: nodes differ for events {np.nonzero((got.node != node).any(1))[0]}"
    assert (_bits32(got.misfit) == _bits32(misfit)).all(), f"{what}: misfit"
    ok = status == api.LOC_OK
    assert (_bits64(got.origin_time[ok]) == _bits64(origin[ok])).all(), f"{what}: origin time"
    assert np.isnan(got.origin_time[~ok]).all() and (got.misfit[~ok] == np.inf).all()


# ---- CPU ---------------------------------------------------------------------------------------

def test_oracle_agrees_with_a_least_squares_fit():
    """The two-pass formula is the residual of min over t0 of sum (obs - tt - t0)^2, which lstsq solves directly."""
    rng = np.random.default_rng(3)
    S, N = 9, 400
    fields = rng.uniform(0, 50, (S, N)).astype(F)
    for e in range(20):
        picks = (fields[:, rng.integers(N)] + F(rng.uniform(-5, 5)) + rng.normal(0, 0.5, S)).astype(F)
        picks[rng.random(S) < 0.2] = np.nan
        mis, t0, k, excl = oracle_misfit(fields, picks)
        keep = ~np.isnan(picks)
        assert k == keep.sum() and not excl.any()
        for n in range(0, N, 37):
            b = picks[keep].astype(np.float64) - fields[keep, n].astype(np.float64)
            x, res, _, _ = np.linalg.lstsq(np.ones((k, 1)), b, rcond=None)
            assert abs(t0[n] - x[0]) <= 1e-12 * max(1.0, abs(x[0]))
            want = float(res[0]) if len(res) else 0.0
            assert abs(float(mis[n]) - want) <= 1e-6 * want + 1e-9, (n, mis[n], want)
    # equal residuals give exactly 0, an infinite time at a picked station excludes the node
    fields[2, 5] = np.inf
    fields[:, 7] = np.arange(S, dtype=F) * F(0.75)   # + 3 is exact
    picks = (fields[:, 7] + F(3)).astype(F)
    picks[4] = np.nan
    mis, t0, k, excl = oracle_misfit(fields, picks)
    assert mis[7] == 0 and t0[7] == 3 and excl[5] and mis[5] == np.inf and excl.sum() == 1


@pytest.mark.skipif(shutil.which("cuobjdump") is None, reason="cuobjdump not on PATH")
def test_locate_kernels_never_fuse_multiply_add():
    out = subprocess.run(["cuobjdump", "-sass", str(P.lib_path())], capture_output=True, text=True, check=True).stdout
    funcs, name = {}, None
    for line in out.splitlines():
        mm = re.search(r"Function : (\S+)", line)
        if mm:
            name = mm.group(1)
            funcs[name] = []
        elif name and re.match(r"\s+/\*[0-9a-f]{4,6}\*/", line):
            funcs[name].append(line)
    kernels = {k: v for k, v in funcs.items() if re.search("locate_kernel|locate_finish|misfit_box", k)}
    assert len(kernels) == 5, sorted(kernels)   # locate_kernel<4, 2, 1>, the finisher, the misfit box
    for k, lines in kernels.items():
        text = "\n".join(lines)
        assert "DADD" in text and "DMUL" in text, k
        assert not re.search(r"\b[DF]FMA2?\b", text), f"{k}: fused multiply-add found"


def test_c99_client_calls_both_location_entry_points(tmp_path):
    """A strict C99 client compiles and links against both entry points.  Without a GPU each fails with a message; with
    one, a tiny constant box and one station: one pick makes every node fit exactly, so the best node is the first."""
    src = tmp_path / "client.c"
    src.write_text(r'''
#include <stdio.h>
#include "sweeptt.h"
int main(void) {
  struct FS fs[7] = {{1, 0, 0, 0.f}, {-1, 0, 0, 0.f}, {0, 1, 0, 0.f}, {0, -1, 0, 0.f}, {0, 0, 1, 0.f},
                     {0, 0, -1, 0.f}, {1, 1, 1, 0.f}};
  struct START st[1] = {{0, 0, 0}}, best[1];
  float v[64], picks[1] = {30.f}, misfit[1], box[64];
  double origin[1];
  int32_t npicks[1], status[1];
  int i;
  sweeptt_stats stats;
  sweeptt_ctx *ctx;
  for (i = 0; i < 64; i++) v[i] = 1.f;
  sweeptt_star_fill_distances(fs, 7, 10.0f);
  ctx = sweeptt_create(NULL);
  if (!ctx) {
    if (sweeptt_locate_events(NULL, 0, 1, picks, 1, best, misfit, origin, npicks, status, &stats)) return 2;
    printf("%s\n", sweeptt_last_error());
    if (sweeptt_misfit_box(NULL, 0, 1, picks, box, &stats)) return 2;
    printf("%s\n", sweeptt_last_error());
    return 0;
  }
  if (!sweeptt_set_model(ctx, v, 4, 4, 4) || !sweeptt_set_star(ctx, fs, 7) || !sweeptt_set_sources(ctx, st, 1) ||
      !sweeptt_run(ctx, NULL) ||
      !sweeptt_locate_events(ctx, 0, 1, picks, 1, best, misfit, origin, npicks, status, &stats) ||
      !sweeptt_misfit_box(ctx, 0, 1, picks, box, &stats)) {
    printf("%s\n", sweeptt_last_error());
    return 3;
  }
  sweeptt_destroy(ctx);
  if (status[0] != SWEEPTT_LOC_OK || npicks[0] != 1 || best[0].i != 0 || best[0].j != 0 || best[0].k != 0) return 4;
  if (misfit[0] != 0.f || origin[0] != 30.0 || box[0] != 0.f || box[63] != 0.f) return 5;
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


# ---- GPU ---------------------------------------------------------------------------------------

DIMS = (21, 18, 16)


def _stations(n, dims=DIMS, seed=0):
    rng = np.random.default_rng(seed)
    flat = rng.choice(int(np.prod(dims)), n, replace=False)
    return np.stack(np.unravel_index(flat, dims), 1).astype(np.int32)


def _events(fields, n, seed, noise=0.05, nan_frac=0.1):
    """Picks [n, S]: the fields at seeded nodes, plus an origin time and noise, with about nan_frac of them NaN."""
    rng = np.random.default_rng(seed)
    S = fields.shape[0]
    flat = fields.reshape(S, -1)
    at = rng.integers(flat.shape[1], size=n)
    picks = (flat[:, at].T + rng.uniform(0, 20, (n, 1)) + rng.normal(0, noise, (n, S))).astype(F)
    picks[rng.random((n, S)) < nan_frac] = np.nan
    return picks


def _context(v, stations, star="818", kernel=None, fields=None):
    ctx = P.SweepContext(kernel=kernel)
    ctx.set_model(v); ctx.set_star(W.star(star)); ctx.set_sources(stations)
    if fields is None:
        ctx.run()
    else:
        for s, f in enumerate(fields):
            ctx.put_tt(s, f)
    return ctx


def _fields(ctx):
    return np.stack([ctx.get_tt(s) for s in range(ctx.nsrc)])


def _check_boxes_and_events(ctx, picks, what):
    fields = _fields(ctx)
    for e in range(min(len(picks), 4)):
        want = oracle_misfit(fields, picks[e])[0]
        got = ctx.misfit_box(picks[e])
        assert (_bits32(got) == _bits32(want)).all(), f"{what}: misfit box of event {e}"
    loc = ctx.locate_events(picks)
    assert_locations_equal(loc, oracle_locate(fields, picks), what)
    assert loc.stats.kernel_launches == 2 and loc.stats.solve_ms > 0
    return fields, loc


@gpu
@pytest.mark.parametrize("kernel", [api.KERNEL_SIMPLE, api.KERNEL_TILED])
@pytest.mark.parametrize("kind", ["random", "hetero", "contrast"])
def test_misfit_box_and_locations_equal_oracle(kind, kernel):
    v = make_field(kind, DIMS, 5)
    stations = _stations(6 + 3 * ["random", "hetero", "contrast"].index(kind), seed=1)
    with _context(v, stations, kernel=kernel) as ctx:
        fields = _fields(ctx)
        picks = _events(fields, 24, seed=2)
        picks[3] = np.nan   # no pick at all
        _check_boxes_and_events(ctx, picks, f"{kind} kernel={kernel}")


@gpu
@pytest.mark.parametrize("axis", ["0", "1", "2"])
def test_locations_do_not_depend_on_the_axis_permutation(axis, monkeypatch):
    monkeypatch.setenv("SWEEPTT_WINDOW_AXIS", axis)
    v = make_field("hetero", DIMS, 6)
    with _context(v, _stations(8, seed=3)) as ctx:
        picks = _events(_fields(ctx), 16, seed=4)
        _check_boxes_and_events(ctx, picks, f"axis {axis}")


@gpu
def test_locations_of_fields_loaded_with_put_tt():
    """Fields put from outside (here: a solve of another model) are used as they are."""
    stations = _stations(7, seed=5)
    with _context(make_field("random", DIMS, 8), stations) as src:
        other = _fields(src)
    with _context(make_field("hetero", DIMS, 9), stations, fields=other) as ctx:
        assert (_bits32(_fields(ctx)) == _bits32(other)).all()
        picks = _events(other, 12, seed=6)
        _check_boxes_and_events(ctx, picks, "put_tt")


@gpu
def test_one_pick_per_event_ties_to_the_first_node():
    """With one pick every reachable node fits exactly (misfit 0): the best node is the smallest caller index."""
    v = make_field("random", DIMS, 11)
    stations = _stations(6, seed=7)
    with _context(v, stations) as ctx:
        fields = _fields(ctx)
        picks = np.full((6, 6), np.nan, F)
        for e in range(6):
            picks[e, e] = F(40 + e)
        loc = ctx.locate_events(picks)
        assert_locations_equal(loc, oracle_locate(fields, picks), "one pick")
        assert (loc.node == 0).all() and (loc.misfit == 0).all() and (loc.npicks == 1).all()
        assert (loc.origin_time == picks[np.arange(6), np.arange(6)].astype(np.float64) - fields[:, 0, 0, 0]).all()


@gpu
def test_mirror_symmetric_stations_tie_to_the_smallest_index():
    dims = (15, 11, 13)
    v = W.constant_field(dims, 0.25)
    stations = np.array([(2, 5, 6), (12, 5, 6), (7, 1, 6), (7, 9, 6)], np.int32)   # mirror pairs about x = 7, y = 5
    with _context(v, stations, star="5") as ctx:
        fields = _fields(ctx)
        # every station is on the plane z = 6, and the 5-FS edge set (its guarded pull included) is symmetric about
        # it: an event at z fits exactly at 12 - z as well
        picks = np.stack([fields[:, 7, 5, 9], fields[:, 4, 3, 8], fields[:, 10, 8, 12]]).astype(F)
        loc = ctx.locate_events(picks)
        assert_locations_equal(loc, oracle_locate(fields, picks), "mirror")
        for e in range(len(picks)):
            box = ctx.misfit_box(picks[e])
            ties = np.argwhere(box == box.min())
            assert box.min() == 0 and len(ties) >= 2, (e, ties)
            assert tuple(loc.node[e]) == tuple(ties[0])


@gpu
def test_an_infinite_wall_leaves_events_unreached():
    """Two stations on either side of an +inf wall thicker than the star's reach share no reachable node: an event
    picked at both is UNREACHED, an event picked at one is located."""
    star = "5"
    reach = int(np.abs(W.star(star)).max())
    dims = (12 + reach + 1, 9, 10)
    v = W.random_field(dims, seed=12)
    v[6:6 + reach + 1] = np.inf
    stations = np.array([(1, 4, 5), (dims[0] - 2, 4, 5)], np.int32)
    with _context(v, stations, star=star) as ctx:
        fields = _fields(ctx)
        assert not (np.isfinite(fields[0]) & np.isfinite(fields[1])).any()
        picks = np.array([[10, 12], [10, np.nan], [np.nan, 7], [np.nan, np.nan]], F)
        loc = ctx.locate_events(picks)
        assert_locations_equal(loc, oracle_locate(fields, picks), "wall")
        assert list(loc.status) == [api.LOC_UNREACHED, api.LOC_OK, api.LOC_OK, api.LOC_NO_PICKS]
        assert (loc.node[[0, 3]] == -1).all() and list(loc.npicks) == [2, 1, 1, 0]
        box = ctx.misfit_box(picks[0])
        assert (box == np.inf).all()


@gpu
def test_noise_free_picks_fit_exactly():
    v = make_field("contrast", DIMS, 13)
    with _context(v, _stations(9, seed=8)) as ctx:
        fields = _fields(ctx)
        rng = np.random.default_rng(9)
        true = rng.integers(int(np.prod(DIMS)), size=30)
        picks = fields.reshape(len(fields), -1)[:, true].T.copy()
        loc = ctx.locate_events(picks)
        assert_locations_equal(loc, oracle_locate(fields, picks), "noise-free")
        assert (loc.status == api.LOC_OK).all() and (loc.misfit == 0).all()
        got = np.ravel_multi_index(tuple(loc.node.T), DIMS)
        assert (got <= true).all()


@gpu
def test_chunks_determinism_and_source_ranges(monkeypatch):
    v = make_field("hetero", DIMS, 14)
    stations = _stations(10, seed=10)
    with _context(v, stations) as ctx:
        fields = _fields(ctx)
        picks = _events(fields, 11, seed=11)
        whole = ctx.locate_events(picks)
        again = ctx.locate_events(picks)
        for f in ("node", "npicks", "status"):
            assert (getattr(whole, f) == getattr(again, f)).all()
        assert (_bits32(whole.misfit) == _bits32(again.misfit)).all()
        assert (_bits64(whole.origin_time) == _bits64(again.origin_time)).all()
        monkeypatch.setenv("SWEEPTT_LOCATE_CHUNK", "3")
        chunked = ctx.locate_events(picks)
        assert chunked.stats.kernel_launches == 4 + 1
        single = [ctx.locate_events(picks[e:e + 1]) for e in range(len(picks))]
        one_by_one = api.Locations(*(np.concatenate([getattr(x, f) for x in single])
                                     for f in ("node", "misfit", "origin_time", "npicks", "status")), None)
        for loc in (chunked, one_by_one):
            assert (loc.node == whole.node).all() and (loc.status == whole.status).all()
            assert (_bits32(loc.misfit) == _bits32(whole.misfit)).all()
            assert (_bits64(loc.origin_time) == _bits64(whole.origin_time)).all()
        monkeypatch.delenv("SWEEPTT_LOCATE_CHUNK")
        sub = picks[:, 2:7]
        loc = ctx.locate_events(sub, sources=(2, 5))
        assert_locations_equal(loc, oracle_locate(fields[2:7], sub), "sources (2, 5)")
        got = ctx.misfit_box(sub[0], sources=range(2, 7))
        assert (_bits32(got) == _bits32(oracle_misfit(fields[2:7], sub[0])[0])).all()
        assert ctx.locate_events(np.zeros((0, 10), F)).status.shape == (0,)


@gpu
def test_refusals_leave_the_context_as_it_was():
    v = make_field("random", DIMS, 15)
    stations = _stations(6, seed=12)
    with _context(v, stations) as ctx:
        fields = _fields(ctx)
        picks = _events(fields, 8, seed=13)
        want = ctx.locate_events(picks)
        pool = ctx.pool_bytes

        def still_the_same(what):
            assert ctx.pool_bytes == pool, what
            got = ctx.locate_events(picks)
            assert (got.node == want.node).all() and (_bits32(got.misfit) == _bits32(want.misfit)).all(), what
            assert (_bits64(got.origin_time) == _bits64(want.origin_time)).all(), what
            assert (_bits32(_fields(ctx)) == _bits32(fields)).all(), what

        for bad in (np.inf, -np.inf):
            p = picks.copy()
            p[5, 2] = bad
            with pytest.raises(P.SweepError, match="INF"):
                ctx.locate_events(p)
            with pytest.raises(P.SweepError, match="INF"):
                ctx.misfit_box(p[5])
            still_the_same(f"pick {bad}")
        with pytest.raises(P.SweepError, match="not within"):
            ctx.locate_events(picks[:, :3], sources=(4, 3))
        with pytest.raises(P.SweepError, match="not within"):
            ctx.misfit_box(picks[0, :0], sources=(0, 0))
        lib = P.load_library()
        p = np.ascontiguousarray(picks)
        node, status = np.empty((8, 3), np.int32), np.empty(8, np.int32)
        assert not lib.sweeptt_locate_events(ctx._h, 0, 6, p.ctypes.data, 8, None, None, None, None,
                                             status.ctypes.data, None)
        assert b"required" in lib.sweeptt_last_error()
        assert not lib.sweeptt_locate_events(ctx._h, 0, 6, p.ctypes.data, 8, node.ctypes.data, None, None, None,
                                             None, None)
        assert not lib.sweeptt_locate_events(ctx._h, 0, 6, None, 8, node.ctypes.data, None, None, None,
                                             status.ctypes.data, None)
        assert not lib.sweeptt_locate_events(ctx._h, 0, 6, p.ctypes.data, -1, node.ctypes.data, None, None, None,
                                             status.ctypes.data, None)
        assert b"negative" in lib.sweeptt_last_error()
        assert not lib.sweeptt_misfit_box(ctx._h, 0, 6, p.ctypes.data, None, None)
        still_the_same("bad arguments")
        # the domain guard: a model whose delays would overflow where the reference's do
        big = v.copy()
        big[3, 3, 3] = F(3e37)
        ctx.set_model(big)
        with pytest.raises(P.SweepError, match="overflows"):
            ctx.locate_events(picks)
        with pytest.raises(P.SweepError, match="overflows"):
            ctx.misfit_box(picks[0])
        ctx.set_model(v)
        ctx.run()
        still_the_same("domain guard")
    with P.SweepContext() as empty:
        with pytest.raises(P.SweepError, match="needs a model"):
            empty.locate_events(picks, sources=(0, 6))
        with pytest.raises(P.SweepError, match="needs a model"):
            empty.misfit_box(picks[0], sources=(0, 6))


@gpu
def test_too_many_stations_for_shared_memory_are_refused():
    """The location kernel stages 32 nodes of every station in shared memory; beyond that the call refuses (the misfit
    box, which reads the fields in place, still works)."""
    dims = (6, 5, 4)
    n = 1000
    starts = np.stack(np.unravel_index(np.arange(n) % 120, dims), 1).astype(np.int32)
    with P.SweepContext() as ctx:
        ctx.set_model(W.random_field(dims, seed=1)); ctx.set_star(W.star("5")); ctx.set_sources(starts)
        ctx.run()
        picks = np.full((1, n), np.nan, F)
        picks[0, :3] = 5
        with pytest.raises(P.SweepError, match="shared memory"):
            ctx.locate_events(picks)
        fields = _fields(ctx)
        assert (_bits32(ctx.misfit_box(picks[0])) == _bits32(oracle_misfit(fields, picks[0])[0])).all()
        for m in (300, 500):   # two and one nodes per thread
            ok = ctx.locate_events(picks[:, :m], sources=(0, m))
            assert_locations_equal(ok, oracle_locate(fields[:m], picks[:, :m]), f"{m} stations")


@gpu
def test_one_shot_locate_events():
    v = make_field("hetero", DIMS, 16)
    stations = _stations(6, seed=14)
    with _context(v, stations) as ctx:
        fields = _fields(ctx)
    picks = _events(fields, 5, seed=15)
    loc = P.locate_events(v, W.star("818"), stations, picks)
    assert_locations_equal(loc, oracle_locate(fields, picks), "one-shot")


@gpu
def test_full_size_config3_exact_picks():
    """config 3: 111 stations (start-111) on the 241x241x51 heterogeneous box; 300 seeded events with exact picks all
    fit exactly, and for four of them the whole misfit box equals the oracle."""
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
        loc = ctx.locate_events(picks)
        assert (loc.status == api.LOC_OK).all() and (loc.misfit == 0).all() and (loc.npicks == 111).all()
        assert (np.ravel_multi_index(tuple(loc.node.T), dims) <= true).all()
        for e in range(4):
            want = oracle_misfit(fields, picks[e])[0]
            got = ctx.misfit_box(picks[e])
            assert (_bits32(got) == _bits32(want)).all(), f"event {e}"
