"""GPU (-m gpu): contexts that live through many calls.  A Gauss-Newton loop keeps one context and changes its model,
star and sources between solves; sweeptt_solve reuses one cached context per device; several contexts share one
device, from one host thread or several.  Between calls a context keeps device state that must follow its inputs
(tensor maps, captured graphs and the wave plan, the host image of the __constant__ star tables and the device-wide
lease on them, tile pull counts, the ray pull table, grow-only buffers).  A missed rebuild gives a plausible field
and no error, so every converged field here is compared bit for bit with the CPU oracle, rays with the ray oracle
and event locations with the location oracle, after every change."""
import functools
import threading

import numpy as np
import pytest

import oracle
import uoparallel_seismic_project_b200 as P
from uoparallel_seismic_project_b200 import api, workloads as W

from conftest import assert_bit_equal, make_field
from test_locate import _events, _stations, assert_locations_equal, oracle_locate
from test_rays import _assert_rays_equal, _one, oracle_rays

pytestmark = pytest.mark.gpu

STARS = {
    "818": W.star("818"),
    "5": W.star("5"),
    "3": W.star("3"),
    # asymmetric subset of the 5-FS star: the generic instantiation of the tiled kernel
    "asym": W.star("5")[np.sort(np.random.default_rng(5).permutation(len(W.star("5")))[:150])],
    # a shorter 818-FS file (its new last entry is the unused one): generic too
    "prefix": W.star("818")[:300],
    # |i| = 9 does not fit the tiled kernel's halo: AUTO falls back to relax_simple
    "wide": np.array([[9, 0, 0], [-9, 0, 0], [0, 1, 0], [0, -1, 0], [0, 0, 1], [0, 0, -1], [1, 1, 1], [-1, -1, -1]],
                     np.int32),
}
KNOBS = ("SWEEPTT_PERSIST", "SWEEPTT_PERSIST_MAX_KEYS", "SWEEPTT_WINDOW_AXIS", "SWEEPTT_WAVE", "SWEEPTT_LOOP",
         "SWEEPTT_GROUPS", "SWEEPTT_BUCKET", "SWEEPTT_LOOKAHEAD", "SWEEPTT_INNER", "SWEEPTT_WAVE_STREAMS")


@pytest.fixture(autouse=True)
def _default_knobs(monkeypatch):
    for k in KNOBS:
        monkeypatch.delenv(k, raising=False)


@functools.lru_cache(maxsize=None)
def _v(kind, dims, seed):
    v = make_field(kind, dims, seed)
    v.flags.writeable = False
    return v


@functools.lru_cache(maxsize=None)
def _ref(case, star, start, used=None):
    """Oracle field of one start on case = (kind, dims, seed); `used` leading entries (None: all but the last)."""
    off = STARS[star] if used is None else STARS[star][: used + 1]
    tt, _, _ = oracle.solve(_v(*case), off, start)
    tt.flags.writeable = False
    return tt


def _kernel_axes(dims, window=None):
    """The kernel's axis order of a caller box, restated from csrc/solver.cu (compute_geometry): the order that wastes
    the fewest lanes at a granularity of 4 x 8 x 8 nodes, ties within 2 % to the caller's order; `window` forces the
    caller axis that becomes the kernel's z.  Used to check the premise of a case, never a result."""
    best, pick = -1.0, None
    for p in ((0, 1, 2), (1, 0, 2), (0, 2, 1), (2, 0, 1), (1, 2, 0), (2, 1, 0)):
        if window is not None and p[2] != window:
            continue
        eff = 1.0
        for q, g in enumerate((4, 8, 8)):
            n = dims[p[q]]
            eff *= n / (-(-n // g) * g)
        if pick is None or eff > best * 1.02:
            best, pick = eff, p
    return pick


def _same_padded_box(a, b):
    """Same kernel axis order and the same 8-node tiles along every axis: the same padded device box."""
    return _kernel_axes(a) == _kernel_axes(b) and all(-(-x // 8) == -(-y // 8) for x, y in zip(a, b))


def _check(ctx, case, star, starts, what, used=None):
    for s, p in enumerate(starts):
        assert_bit_equal(ctx.get_tt(s), _ref(case, star, tuple(p), used), f"{what}: source {s} at {p}")
        assert ctx.count_violations(s) == 0, f"{what}: source {s} violates the fixed point"


def _receivers(dims, n=20, seed=0):
    rng = np.random.default_rng(seed)
    corners = [(x, y, z) for x in (0, dims[0] - 1) for y in (0, dims[1] - 1) for z in (0, dims[2] - 1)]
    return np.concatenate([corners, np.stack([rng.integers(0, d, n) for d in dims], 1)]).astype(np.int32)


def _check_rays(ctx, case, star, starts, what):
    rec = _receivers(case[1])
    rays = ctx.trace_rays(rec)
    for s, p in enumerate(starts):
        want = oracle_rays(_v(*case), _ref(case, star, tuple(p)), STARS[star], p, rec)
        _assert_rays_equal(_one(rays, s), want, f"{what}: rays of source {s}")


def _check_locate(ctx, case, star, starts, what, seed=0):
    fields = np.stack([_ref(case, star, tuple(p)) for p in starts])
    picks = _events(fields, 8, seed=seed)
    assert_locations_equal(ctx.locate_events(picks), oracle_locate(fields, picks), f"{what}: locations")


def _context(case, star, starts, **kw):
    ctx = P.SweepContext(**kw)
    ctx.set_model(_v(*case)); ctx.set_star(STARS[star]); ctx.set_sources(starts)
    return ctx


# ---- 1. one context through a script of changes ---------------------------------------------------------------------

def test_one_context_through_a_script_of_changes(monkeypatch):
    dims = (29, 24, 24)
    a, a2 = ("hetero", dims, 3), ("random", dims, 4)
    narrow = ("hetero", (27, 24, 24), 5)            # a new nx in the same padded box: only the x clipping changes
    big = ("contrast", (36, 30, 26), 6)              # a larger padded box
    assert _kernel_axes(dims) == (0, 1, 2) and _same_padded_box(dims, narrow[1])
    assert not _same_padded_box(dims, big[1]) and _kernel_axes(big[1])[2] != 0
    s3 = [(3, 4, 5), (26, 23, 0), (14, 2, 23)]
    s5 = s3 + [(0, 0, 0), (20, 12, 11)]
    with P.SweepContext() as ctx:
        ctx.set_model(_v(*a)); ctx.set_star(STARS["818"]); ctx.set_sources(s3)
        assert ctx.run().kernel_used == api.KERNEL_TILED
        _check(ctx, a, "818", s3, "first solve")
        _check_rays(ctx, a, "818", s3, "first solve")
        _check_locate(ctx, a, "818", s3, "first solve")

        ctx.set_model(_v(*a2))                      # model update: star and sources kept
        ctx.run()
        _check(ctx, a2, "818", s3, "model update")
        _check_rays(ctx, a2, "818", s3, "model update")
        _check_locate(ctx, a2, "818", s3, "model update", seed=1)

        # more sources than one single-launch solve holds: waves of 2 + 2 + 1, then back to one source
        monkeypatch.setenv("SWEEPTT_PERSIST", "1")
        monkeypatch.setenv("SWEEPTT_PERSIST_MAX_KEYS", str(2 * ctx.tiles_per_source + 1))
        ctx.set_sources(s5)
        assert ctx.run().relax_launches == 3
        _check(ctx, a2, "818", s5, "5 sources in waves")
        monkeypatch.delenv("SWEEPTT_PERSIST_MAX_KEYS")
        ctx.set_sources(s5[:1])
        assert ctx.run().relax_launches == 1
        _check(ctx, a2, "818", s5[:1], "back to one source")
        monkeypatch.delenv("SWEEPTT_PERSIST")

        # stars: RXY, the stock kernel, the scheduler and the kernel choice move back and forth
        ctx.set_sources(s3)
        for star in ("5", "3", "asym", "wide", "818"):
            ctx.set_star(STARS[star])
            st = ctx.run()
            assert st.kernel_used == (api.KERNEL_SIMPLE if star == "wide" else api.KERNEL_TILED), star
            _check(ctx, a2, star, s3, f"star {star}")
            _check_rays(ctx, a2, star, s3, f"star {star}")
            _check_locate(ctx, a2, star, s3, f"star {star}", seed=2)

        ctx.set_model(_v(*narrow))                  # sources still inside: kept
        ctx.run()
        _check(ctx, narrow, "818", s3, "new nx")
        _check_rays(ctx, narrow, "818", s3, "new nx")

        ctx.set_model(_v(*big))                     # a new padded box drops the sources
        with pytest.raises(P.SweepError, match="start points"):
            ctx.run()
        ctx.set_sources(s3)
        ctx.run()
        _check(ctx, big, "818", s3, "larger box")

        monkeypatch.setenv("SWEEPTT_WINDOW_AXIS", "0")  # a new axis order drops the sources too
        ctx.set_model(_v(*big))
        with pytest.raises(P.SweepError, match="start points"):
            ctx.run()
        ctx.set_sources(s3)
        ctx.run()
        _check(ctx, big, "818", s3, "new axis order")
        _check_rays(ctx, big, "818", s3, "new axis order")
        _check_locate(ctx, big, "818", s3, "new axis order", seed=3)
        monkeypatch.delenv("SWEEPTT_WINDOW_AXIS")

        ctx.reset()                                 # a partly relaxed field, then a new star and a fresh run
        ctx.step(1)
        ctx.set_star(STARS["5"])
        ctx.run()
        _check(ctx, big, "5", s3, "step, set_star, run")

        # a partly swept oracle state under a new star, relaxed from there with step()
        ctx.set_star(STARS["3"])
        for s, p in enumerate(s3):
            part, _, _ = oracle.solve(_v(*big), STARS["3"], p, maxsweeps=1)
            assert not np.array_equal(part, _ref(big, "3", p))
            ctx.put_tt(s, part)
        for _ in range(1000):
            if not ctx.step(4)[0]:
                break
        _check(ctx, big, "3", s3, "put_tt, then step")


# ---- 2. start points that a new model leaves outside ------------------------------------------------------------------

@pytest.mark.parametrize("axis,n", [(0, 25), (1, 29), (2, 29)])
def test_a_model_that_leaves_a_start_point_outside_drops_the_sources(axis, n):
    """32 -> n along one axis keeps the padded box and the axis order, but the start at 31 is now in the +INF padding:
    the context must drop its start points (as sweeptt_set_sources would refuse that one), not return an all-INF
    field."""
    base = (32, 32, 32)
    small = tuple(n if q == axis else d for q, d in enumerate(base))
    assert _same_padded_box(base, small)
    out = tuple(31 if q == axis else 5 for q in range(3))
    full, shrunk = ("hetero", base, 7), ("hetero", small, 8)
    with _context(full, "5", [out, (3, 4, 5)]) as ctx:
        ctx.run()
        _check(ctx, full, "5", [out, (3, 4, 5)], "before")
        ctx.set_model(_v(*shrunk))
        with pytest.raises(P.SweepError, match="start points"):
            ctx.run()
        with pytest.raises(P.SweepError, match="outside"):
            ctx.set_sources([out])
        ctx.set_sources([(3, 4, 5)])
        ctx.run()
        _check(ctx, shrunk, "5", [(3, 4, 5)], "after set_sources")


def test_a_model_that_keeps_every_start_point_inside_keeps_them():
    base, small = (32, 32, 32), (29, 32, 30)
    assert _same_padded_box(base, small)
    starts = [(28, 31, 29), (0, 5, 7)]
    full, shrunk = ("random", base, 9), ("random", small, 10)
    with _context(full, "5", starts) as ctx:
        ctx.run()
        ctx.set_model(_v(*shrunk))
        ctx.run()
        _check(ctx, shrunk, "5", starts, "shrunk, sources kept")
        bad = np.array(_v(*full))
        bad[31, 31, 31] = np.nan
        with pytest.raises(P.SweepError, match="NaN"):
            ctx.set_model(bad)                          # a refused model changes nothing, sources included
        ctx.run()
        _check(ctx, shrunk, "5", starts, "after a refused model")


# ---- 3. several contexts on one device, one thread --------------------------------------------------------------------

def test_interleaved_contexts_on_one_device_take_turns_on_the_star_tables():
    box1, box2 = ("hetero", (29, 24, 24), 11), ("random", (24, 31, 20), 12)
    box1_nx = ("hetero", (27, 24, 24), 13)          # same star, another x extent: another __constant__ image
    wide_box, solve_box = ("contrast", (26, 14, 12), 14), ("hetero", (20, 22, 18), 15)
    cases = {"A": (box1, "818", [(3, 4, 5), (28, 0, 23)]), "B": (box2, "5", [(12, 30, 0)]),
             "C": (box1_nx, "818", [(20, 10, 10)]), "D": (box2, "asym", [(1, 2, 3), (23, 15, 19)]),
             "E": (wide_box, "wide", [(12, 7, 6)])}
    ctx = {k: _context(case, star, starts) for k, (case, star, starts) in cases.items()}
    solve_starts = [(10, 11, 9), (0, 0, 0)]

    def solve_sixth():
        tt, _ = P.solve(_v(*solve_box), STARS["prefix"], solve_starts)
        for s, p in enumerate(solve_starts):
            assert_bit_equal(tt[s], _ref(solve_box, "prefix", p), f"sweeptt_solve source {s}")

    def run(k):
        def go():
            case, star, starts = cases[k]
            ctx[k].run()
            _check(ctx[k], case, star, starts, f"context {k}")
        return go

    try:
        others = [run("B"), run("C"), solve_sixth, run("D"), run("E")]
        ctx["A"].reset()
        for other in others * 2:                    # every step of A takes the lease back from another star
            ctx["A"].step(1)
            other()
        for _ in range(1000):
            if not ctx["A"].step(2)[0]:
                break
        for k, (case, star, starts) in cases.items():
            _check(ctx[k], case, star, starts, f"context {k} at the end")
        _check_rays(ctx["A"], *cases["A"], "context A")
        _check_rays(ctx["C"], *cases["C"], "context C")
        _check_locate(ctx["D"], *cases["D"], "context D")
    finally:
        for c in ctx.values():
            c.close()
        P.load_library().sweeptt_release_cache()


# ---- 4. several host threads ------------------------------------------------------------------------------------------

def _run_threads(jobs, timeout=300):
    """Runs every job in its own daemon thread, started together on a barrier.  A thread still alive after the
    timeout (a deadlock) fails the test instead of hanging it; an exception in a thread fails it too."""
    barrier = threading.Barrier(len(jobs))
    errors = {}

    def wrap(name, fn):
        try:
            barrier.wait(timeout)
            fn()
        except BaseException as e:  # noqa: BLE001 (reported below)
            errors[name] = e

    threads = [threading.Thread(target=wrap, args=(n, f), name=n, daemon=True) for n, f in jobs.items()]
    for t in threads:
        t.start()
    for t in threads:
        t.join(timeout)
    alive = [t.name for t in threads if t.is_alive()]
    assert not alive, f"threads still running after {timeout} s: {alive}"
    for name, e in errors.items():
        raise AssertionError(f"thread {name}: {e!r}") from e


def test_host_threads_each_with_its_own_context_equal_the_oracle():
    ctx_cases = {  # star -> (kind, dims, starts); three models per thread (seeds 0, 1, 2)
        "818": ("hetero", (29, 24, 24), [(3, 4, 5), (26, 20, 1)]),
        "5": ("random", (24, 31, 20), [(12, 30, 0)]),
        "3": ("contrast", (36, 20, 25), [(35, 0, 24), (1, 1, 1)]),
        "asym": ("hetero", (20, 33, 24), [(10, 16, 12)]),
        "wide": ("random", (26, 14, 12), [(12, 7, 6)]),
    }
    solve_cases = {"818": ("random", (22, 25, 19), [(1, 2, 3), (21, 24, 18)]),
                   "5": ("hetero", (30, 18, 21), [(15, 9, 10)])}
    for cases in (ctx_cases, solve_cases):          # the oracle first, in this thread
        for star, (kind, dims, starts) in cases.items():
            for it in range(3):
                for p in starts:
                    _ref((kind, dims, 30 + it), star, p)
    got = {}

    def context_job(star, kind, dims, starts):
        def job():
            with P.SweepContext() as c:
                c.set_star(STARS[star])
                for it in range(3):
                    c.set_model(_v(kind, dims, 30 + it))
                    if it == 0:
                        c.set_sources(starts)
                    c.run()
                    got[("ctx", star, it)] = [c.get_tt(s) for s in range(len(starts))]
        return job

    def solve_job(star, kind, dims, starts):
        def job():
            for it in range(3):
                got[("solve", star, it)] = list(P.solve(_v(kind, dims, 30 + it), STARS[star], starts)[0])
        return job

    # event location takes the lease too: its own context and star, single-threaded results first
    loc_case, stations = ("hetero", (21, 18, 16), 40), _stations(6, (21, 18, 16), seed=1)
    loc_ctx = _context(loc_case, "3", stations)
    try:
        loc_ctx.run()
        _check(loc_ctx, loc_case, "3", stations, "location context")
        fields = np.stack([loc_ctx.get_tt(s) for s in range(len(stations))])
        picks = _events(fields, 12, seed=4)
        want_loc = loc_ctx.locate_events(picks)
        assert_locations_equal(want_loc, oracle_locate(fields, picks), "single-threaded")
        levels = np.where(want_loc.status == api.LOC_OK, want_loc.misfit + np.float32(4), np.nan).astype(np.float32)
        want_reg = loc_ctx.misfit_regions(picks, levels)

        def locate_job():
            for it in range(3):
                got[("loc", it)] = (loc_ctx.locate_events(picks), loc_ctx.misfit_regions(picks, levels))

        jobs = {f"context {s}": context_job(s, *c) for s, c in ctx_cases.items()}
        jobs.update({f"solve {s}": solve_job(s, *c) for s, c in solve_cases.items()})
        jobs["locate"] = locate_job
        _run_threads(jobs)
    finally:
        loc_ctx.close()
        P.load_library().sweeptt_release_cache()

    for kind_of, cases in (("ctx", ctx_cases), ("solve", solve_cases)):
        for star, (kind, dims, starts) in cases.items():
            for it in range(3):
                for s, p in enumerate(starts):
                    assert_bit_equal(got[(kind_of, star, it)][s], _ref((kind, dims, 30 + it), star, p),
                                     f"{kind_of} thread {star}, iteration {it}, source {s}")
    for it in range(3):
        loc, reg = got[("loc", it)]
        assert_locations_equal(loc, oracle_locate(fields, picks), f"locate thread, iteration {it}")
        for f in ("count", "lo", "hi", "moments", "npicks", "status"):
            assert (getattr(reg, f) == getattr(want_reg, f)).all(), f"misfit_regions {f}, iteration {it}"
        for f in ("origin_min", "origin_max"):
            a, b = getattr(reg, f), getattr(want_reg, f)
            assert (a.view(np.uint64) == b.view(np.uint64)).all(), f"misfit_regions {f}, iteration {it}"


# ---- 5. sweeptt_solve's cached context across options --------------------------------------------------------------

def test_the_cached_context_follows_every_option(monkeypatch):
    box, other = ("hetero", (29, 24, 24), 50), ("random", (33, 21, 27), 51)
    starts = [(3, 4, 5), (28, 23, 23)]

    def solve(case, star, pts, used=None, **opts):
        tt, st = P.solve(_v(*case), STARS[star], pts, star_used=used, **opts)
        for s, p in enumerate(pts):
            assert_bit_equal(tt[s], _ref(case, star, tuple(p), used), f"{opts} star_used={used}: source {s}")
        return st

    try:
        assert solve(box, "818", starts, kernel=api.KERNEL_SIMPLE).kernel_used == api.KERNEL_SIMPLE
        assert solve(box, "818", starts, kernel=api.KERNEL_TILED).kernel_used == api.KERNEL_TILED
        assert solve(box, "818", starts, kernel=api.KERNEL_AUTO).kernel_used == api.KERNEL_TILED
        solve(box, "818", starts, loop=api.LOOP_BATCHED)
        solve(box, "818", starts, loop=api.LOOP_GRAPH)
        solve(box, "818", starts, max_rounds=100000)
        solve(box, "818", starts, max_rounds=0)
        solve(box, "818", starts, used=300)         # the first 300 entries only: the star tables must follow
        solve(box, "818", starts)                   # and back to all but the last
        solve(box, "5", starts, used=100)
        solve(box, "5", starts)
        # another box, star and source count, across waves and back
        with P.SweepContext() as probe:
            probe.set_model(_v(*other)); probe.set_star(STARS["3"]); probe.set_sources(starts[:1])
            ntiles = probe.tiles_per_source
        many = [(0, 0, 0), (32, 20, 26), (16, 10, 13), (5, 19, 2), (30, 1, 25)]
        monkeypatch.setenv("SWEEPTT_PERSIST", "1")
        monkeypatch.setenv("SWEEPTT_PERSIST_MAX_KEYS", str(2 * ntiles + 1))
        assert solve(other, "3", many).relax_launches == 3
        monkeypatch.delenv("SWEEPTT_PERSIST_MAX_KEYS")
        monkeypatch.delenv("SWEEPTT_PERSIST")
        solve(other, "asym", many[:1])
        solve(box, "818", starts)
    finally:
        P.load_library().sweeptt_release_cache()


# ---- 6. two devices -------------------------------------------------------------------------------------------------

def _need(n):
    have = P.device_count()
    if have < n:
        pytest.skip(f"needs {n} GPUs, this box has {have}")


def test_contexts_on_two_devices_equal_device_0():
    _need(2)
    case, star, starts = ("hetero", (29, 24, 24), 60), "818", [(3, 4, 5), (26, 20, 1)]
    case5, starts5 = ("random", (24, 31, 20), 61), [(12, 30, 0), (0, 0, 19)]
    models = {"818": case, "5": case5}
    ctx = {(d, k): _context(c, s, p, device=d) for d in (0, 1)
           for k, (c, s, p) in {"818": (case, star, starts), "5": (case5, "5", starts5)}.items()}
    rec = _receivers(case[1])
    try:
        out = {}
        for d, k in ((0, "818"), (1, "818"), (1, "5"), (0, "5")):     # one thread, interleaved
            ctx[(d, k)].run()
            out[(d, k)] = [ctx[(d, k)].get_tt(s) for s in range(2)]
        for k in ("818", "5"):
            for s in range(2):
                assert_bit_equal(out[(1, k)][s], out[(0, k)][s], f"{k}: device 1 vs 0, source {s}")
        _check(ctx[(0, "818")], case, star, starts, "device 0")
        r0, r1 = ctx[(0, "818")].trace_rays(rec), ctx[(1, "818")].trace_rays(rec)
        for s in range(2):
            _assert_rays_equal(_one(r1, s), _one(r0, s), f"rays, device 1 vs 0, source {s}")
        fields = np.stack(out[(0, "5")])
        picks = _events(fields, 8, seed=5)
        assert_locations_equal(ctx[(1, "5")].locate_events(picks), oracle_locate(fields, picks), "locate on device 1")

        def job(d):
            def go():
                for it in range(3):
                    for k in ("818", "5"):
                        ctx[(d, k)].set_model(_v(models[k][0], models[k][1], 70 + it))
                        ctx[(d, k)].run()
                        out[(d, k, it)] = [ctx[(d, k)].get_tt(s) for s in range(2)]
            return go

        _run_threads({"device 0": job(0), "device 1": job(1)})
        for it in range(3):
            for k in ("818", "5"):
                for s in range(2):
                    assert_bit_equal(out[(1, k, it)][s], out[(0, k, it)][s], f"threads, {k}, iteration {it}, source {s}")
        for s, p in enumerate(starts):
            assert_bit_equal(out[(1, "818", 2)][s], _ref(("hetero", case[1], 72), star, p), f"device 1 vs oracle {s}")
    finally:
        for c in ctx.values():
            c.close()
