"""The sweep at the float edges of its inputs (DESIGN §1, include/sweeptt.h).

The kernels evaluate an edge delay as fl(hd * fl(v_n + v_m)) with hd = fl(0.5f * d); the reference as
fl(fl(d * fl(v_n + v_m)) / 2.0).  The two agree on a domain that ready() guards:
  fl(dmax * fl(vmax + vmax)) finite,  every positive d >= 2^-125,  fl(dpos * vpos) >= 2^-125.
Outside it a run is refused; negative, NaN or infinite star distances and negative or NaN slowness are refused by
set_star / set_model, and a refused call leaves the context as it was.

CPU: the domain claim in numpy over every float32 binade (and a mismatch just outside each bound); the oracle's field
does not depend on the sign of a zero slowness.  GPU (-m gpu): every field equals the oracle's bit for bit, with no
violations, for -0.0 / +0.0 regions (every scheduler, slabs), +INF walls and starts, non-default delta, slowness over
60 decades, models on the last accepted float of each bound; the refusals at every entry point; rays on a
signed-zero model."""
import functools

import numpy as np
import pytest

import oracle
import uoparallel_seismic_project_b200 as P
from uoparallel_seismic_project_b200 import api, workloads as W

from conftest import assert_bit_equal
from test_rays import _assert_rays_equal, all_nodes, oracle_rays

gpu = pytest.mark.gpu
F = np.float32
LO = F(2.0 ** -125)
FLT_MAX = np.finfo(np.float32).max
STALLED = api.RAY_STALLED
STARS = ("3", "5", "818")
DELTAS = (10.0, 1.0, 0.3, 2.5, 1e-3, 1e3)
MODES = {  # (kernel, environment)
    "simple": (api.KERNEL_SIMPLE, {}),
    "tiled_rounds": (api.KERNEL_TILED, {"SWEEPTT_PERSIST": "0"}),
    "tiled_persistent": (api.KERNEL_TILED, {"SWEEPTT_PERSIST": "1"}),
}


# ---- the two delay forms and the guard, restated in numpy ---------------------------------------

def kernel_delay(d, va, vb):
    """fl(fl(0.5f * d) * fl(va + vb)): the kernels' expression."""
    with np.errstate(all="ignore"):
        return (F(0.5) * F(d)) * (F(va) + F(vb))


def reference_delay(d, va, vb):
    """(float)((double)fl(d * fl(va + vb)) / 2.0): the reference's expression (oracle/sweep_oracle.c)."""
    with np.errstate(all="ignore"):
        return (np.float64(F(d) * (F(va) + F(vb))) / 2.0).astype(F)


def star_range(off, delta):
    """(dmax, dpos) over the star's used entries (all but the last, self edges skipped), d computed like make_star."""
    off = np.asarray(off, np.int32)
    d = oracle.star_distances(off, delta)[:-1][(off[:-1] != 0).any(1)]
    pos = d[d > 0]
    return F(d.max()), (F(pos.min()) if len(pos) else F(np.inf))


def model_range(v):
    """(vmax, vpos): the largest finite and the smallest positive slowness (+INF if none)."""
    v = np.asarray(v, F)
    fin = v[np.isfinite(v)]
    pos = v[v > 0]
    return (F(fin.max()) if len(fin) else F(0)), (F(pos.min()) if len(pos) else F(np.inf))


def guard_accepts(dmax, dpos, vmax, vpos):
    with np.errstate(all="ignore"):
        return bool(np.isfinite(F(dmax) * (F(vmax) + F(vmax))) and F(dpos) >= LO and F(dpos) * F(vpos) >= LO)


def _bisect_float(pred, lo_bits, hi_bits):
    """Smallest float32 bit pattern in (lo_bits, hi_bits] for which the monotone pred holds (pred(hi) is True)."""
    while hi_bits - lo_bits > 1:
        mid = (lo_bits + hi_bits) // 2
        if pred(np.uint32(mid).view(F)):
            hi_bits = mid
        else:
            lo_bits = mid
    return np.uint32(hi_bits).view(F)


def last_vmax(dmax):
    """The largest slowness the overflow bound accepts with this dmax."""
    over = lambda v: not np.isfinite(kernel_delay(F(2) * F(dmax), v, v))  # fl(dmax * fl(v + v)), hd = dmax exactly
    first_bad = _bisect_float(over, 0, 0x7f800000)
    return np.nextafter(first_bad, F(0))


def first_vpos(dpos):
    """The smallest positive slowness the subnormal bound accepts with this dpos."""
    with np.errstate(all="ignore"):
        return _bisect_float(lambda v: F(dpos) * v >= LO, 0, 0x7f800000)


def _binade_values(seed=0, per=3):
    """Non-negative float32 values in every binade (subnormals included), around FLT_MAX, and the specials."""
    rng = np.random.default_rng(seed)
    mant = rng.integers(0, 1 << 23, size=(255, per), dtype=np.uint32)
    normal = ((np.arange(1, 255, dtype=np.uint32)[:, None] << 23) | mant[:254]).ravel().view(F)
    sub = (rng.integers(1, 1 << 23, size=40, dtype=np.uint32)).view(F)
    top = np.array([FLT_MAX, np.nextafter(FLT_MAX, F(0)), FLT_MAX / 2, np.nextafter(FLT_MAX / 2, F(np.inf))], F)
    special = np.array([0.0, -0.0, np.inf, 2.0 ** -149, 2.0 ** -126, LO], F)
    return np.concatenate([normal, sub, top, special]).astype(F)


# ---- CPU: the domain claim ----------------------------------------------------------------------

@pytest.mark.parametrize("name", STARS)
def test_the_two_delay_forms_agree_wherever_the_guard_accepts(name):
    """Every pair (va, vb) of values from every binade is a two-node model; for every distinct d of the star the
    guard's verdict on that model and star implies fl(fl(0.5f*d)*s) == (float)((double)fl(d*s)/2.0)."""
    off = W.star(name)
    vals = _binade_values(seed=1)
    va, vb = np.meshgrid(vals, vals, indexing="ij")
    va, vb = va.ravel(), vb.ravel()
    with np.errstate(all="ignore"):
        vmax = np.maximum(np.where(np.isfinite(va), va, 0), np.where(np.isfinite(vb), vb, 0)).astype(F)
        pa, pb = np.where(va > 0, va, np.inf), np.where(vb > 0, vb, np.inf)
        vpos = np.minimum(pa, pb).astype(F)
    accepted_total = 0
    for delta in DELTAS:
        dmax, dpos = star_range(off, delta)
        d_all = np.unique(oracle.star_distances(off, delta)[:-1][(off[:-1] != 0).any(1)])
        with np.errstate(all="ignore"):
            ok = np.isfinite(dmax * (vmax + vmax)) & (dpos >= LO) & (dpos * vpos >= LO)
        assert ok.any()
        accepted_total += int(ok.sum())
        for d in d_all:
            k = kernel_delay(d, va[ok], vb[ok])
            r = reference_delay(d, va[ok], vb[ok])
            same = (k.view(np.uint32) == r.view(np.uint32)) | (np.isnan(k) & np.isnan(r))
            assert same.all(), (f"delta {delta}, d {d}: {int((~same).sum())} accepted pairs differ, e.g. "
                                f"va={va[ok][~same][0]!r} vb={vb[ok][~same][0]!r}")
    assert accepted_total > len(va)  # (the accepted pairs span the binades, not a corner)


@pytest.mark.parametrize("name", STARS)
def test_just_beyond_the_overflow_bound_the_forms_differ(name):
    off = W.star(name)
    checked = 0
    for delta in DELTAS:
        dmax, dpos = star_range(off, delta)
        v = last_vmax(dmax)
        assert guard_accepts(dmax, dpos, v, F(1))
        assert kernel_delay(dmax, v, v) == reference_delay(dmax, v, v)
        beyond = np.nextafter(v, F(np.inf))
        assert not guard_accepts(dmax, dpos, beyond, F(1))
        if dmax > 1:  # (with dmax <= 1 only an infinite v + v overflows d * (v + v), and then both forms are inf)
            assert np.isinf(reference_delay(dmax, beyond, beyond)) and np.isfinite(kernel_delay(dmax, beyond, beyond))
            checked += 1
    assert checked >= 3


def test_just_below_the_distance_bound_half_d_rounds():
    for d in (np.nextafter(LO, F(0)), F(3 * 2.0 ** -149), np.nextafter(LO / 2, F(0))):
        assert not guard_accepts(d, d, F(1), F(1))
        s = np.float32(2.0 ** 60)
        assert kernel_delay(d, s, F(0)) != reference_delay(d, s, F(0)), d
    assert guard_accepts(LO, LO, F(1), F(1))
    assert kernel_delay(LO, F(2.0 ** 60), F(0)) == reference_delay(LO, F(2.0 ** 60), F(0))


@pytest.mark.parametrize("name", STARS)
def test_just_below_the_subnormal_bound_the_reference_rounds_twice(name):
    off = W.star(name)
    rng = np.random.default_rng(2)
    dmax, dpos = star_range(off, 10.0)
    first = first_vpos(dpos)
    assert guard_accepts(dmax, dpos, F(1), first) and not guard_accepts(dmax, dpos, F(1), np.nextafter(first, F(0)))
    d_all = np.unique(oracle.star_distances(off, 10.0)[:-1][(off[:-1] != 0).any(1)])
    below = rng.integers(1, first.view(np.uint32), size=200000, dtype=np.uint32).view(F)
    mismatches = 0
    for d in d_all:
        mismatches += int((kernel_delay(d, below, F(0)) != reference_delay(d, below, F(0))).sum())
        bound = first_vpos(d)  # from d's own bound up, the forms agree
        v = (bound.view(np.uint32) + np.arange(0, 1 << 16, dtype=np.uint32)).view(F)
        assert (kernel_delay(d, v, F(0)).view(np.uint32) == reference_delay(d, v, F(0)).view(np.uint32)).all(), d
    assert mismatches > 0


# ---- models -------------------------------------------------------------------------------------

DIMS = (24, 20, 18)


def _signed_zero_models():
    """name -> (model with -0.0 and no +0.0, starts: inside a zero region, outside one, on its boundary)."""
    v = np.full(DIMS, 0.3, F)
    slab = v.copy()
    slab[8:12] = -0.0
    x, y, z = np.indices(DIMS)
    blob = v.copy()
    c = (12, 9, 8)
    blob[(x - c[0]) ** 2 + (y - c[1]) ** 2 + (z - c[2]) ** 2 <= 25] = -0.0
    island = np.full(DIMS, -0.0, F)
    island[14:21, 3:12, 5:15] = W.random_field((7, 9, 10), seed=4)
    return {
        "slab": (slab, [(10, 5, 5), (2, 10, 9), (8, 3, 12)]),
        "blob": (blob, [c, (0, 19, 0), (17, 9, 8)]),
        "island": (island, [(1, 1, 1), (17, 7, 9), (14, 3, 5)]),
    }


def _twin(v):
    """The same model with every zero +0.0."""
    return np.where(v == 0, F(0.0), v).astype(F)


@functools.lru_cache(maxsize=None)
def _oracle_zero(model, star, start, sign):
    v, _ = _signed_zero_models()[model]
    return oracle.solve(v if sign < 0 else _twin(v), W.star(star), start)[0]


# ---- CPU: oracle metamorphic checks -------------------------------------------------------------

@pytest.mark.parametrize("name", STARS)
def test_oracle_field_does_not_depend_on_the_sign_of_zero(name):
    for model, (v, starts) in _signed_zero_models().items():
        assert (v == 0).any() and not (np.signbit(v) == 0)[v == 0].any()  # -0.0 only
        zero_reach = 0
        for s in starts:
            a, b = _oracle_zero(model, name, s, -1), _oracle_zero(model, name, s, +1)
            assert_bit_equal(a, b, f"{model} from {s}")
            zero_reach += int((a == 0).sum()) - 1
        assert zero_reach > 0, model  # zero-delay edges carry time 0 beyond a start


# ---- GPU helpers --------------------------------------------------------------------------------

def _env(monkeypatch, env):
    for k in ("SWEEPTT_PERSIST", "SWEEPTT_PERSIST_MAX_KEYS", "SWEEPTT_WAVE"):
        monkeypatch.delenv(k, raising=False)
    for k, val in env.items():
        monkeypatch.setenv(k, str(val))


def _ctx_solve(v, star, starts, delta=10.0, kernel=None):
    """(fields, violations, stats) from one context."""
    with P.SweepContext(kernel=kernel) as ctx:
        ctx.set_model(v); ctx.set_star(star, delta); ctx.set_sources(starts)
        st = ctx.run()
        return [ctx.get_tt(s) for s in range(len(starts))], [ctx.count_violations(s) for s in range(len(starts))], st


def _check_against_oracle(v, name, starts, delta=10.0, kernel=None, what=""):
    tts, viol, st = _ctx_solve(v, W.star(name), starts, delta, kernel)
    assert viol == [0] * len(starts), f"{what}: violations {viol}"
    for s, p in enumerate(starts):
        ref, _, _ = oracle.solve(v, W.star(name), p, delta=delta)
        assert_bit_equal(tts[s], ref, f"{what} from {p}")
    return tts, st


# ---- GPU: signed zero ---------------------------------------------------------------------------

@gpu
@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("name", STARS)
def test_negative_zero_slowness_equals_positive_zero(name, mode, monkeypatch):
    kernel, env = MODES[mode]
    _env(monkeypatch, env)
    for model, (v, starts) in _signed_zero_models().items():
        neg, vn, _ = _ctx_solve(v, W.star(name), starts, kernel=kernel)
        pos, vp, _ = _ctx_solve(_twin(v), W.star(name), starts, kernel=kernel)
        assert vn == [0] * 3 and vp == [0] * 3, (model, vn, vp)
        for s, p in enumerate(starts):
            ref = _oracle_zero(model, name, p, -1)
            assert_bit_equal(neg[s], ref, f"{model} -0.0 from {p}")
            assert_bit_equal(pos[s], neg[s], f"{model} +0.0 twin from {p}")


@gpu
@pytest.mark.parametrize("name", ["5", "818"])
def test_negative_zero_in_waves_of_single_launches(name, monkeypatch):
    v, starts = _signed_zero_models()["slab"]
    _env(monkeypatch, {})
    with P.SweepContext(kernel=api.KERNEL_TILED) as probe:
        probe.set_model(v); probe.set_star(W.star(name)); probe.set_sources(starts[:1])
        ntiles = probe.tiles_per_source
    _env(monkeypatch, {"SWEEPTT_PERSIST": 1, "SWEEPTT_PERSIST_MAX_KEYS": 2 * ntiles + 1})
    tts, viol, st = _ctx_solve(v, W.star(name), starts, kernel=api.KERNEL_TILED)
    assert st.relax_launches == 2 and viol == [0] * 3
    for s, p in enumerate(starts):
        assert_bit_equal(tts[s], _oracle_zero("slab", name, p, -1), f"waves from {p}")


@gpu
@pytest.mark.parametrize("slabs", [2, 3])
@pytest.mark.parametrize("name", ["5", "818"])
def test_negative_zero_over_slabs(name, slabs):
    for model, (v, starts) in _signed_zero_models().items():
        for p in starts:
            tt, _ = P.solve_slabs(v, W.star(name), p, num_slabs=slabs, slab_axis=0)
            assert_bit_equal(tt, _oracle_zero(model, name, p, -1), f"{model} over {slabs} slabs from {p}")


@gpu
def test_rays_on_a_signed_zero_model_equal_oracle_rays():
    v, starts = _signed_zero_models()["slab"]
    off = W.star("5")
    rec = all_nodes(DIMS)
    with P.SweepContext() as ctx:
        ctx.set_model(v); ctx.set_star(off); ctx.set_sources(starts)
        ctx.run()
        rays = ctx.trace_rays(rec)
    stalled = 0
    for s, p in enumerate(starts):
        want = oracle_rays(v, _oracle_zero("slab", "5", p, -1), off, p, rec)
        _assert_rays_equal((rays.nodes[s], rays.length[s], rays.status[s], rays.tt[s]), want, f"from {p}")
        stalled += int((want[2] == STALLED).sum())
    assert stalled > 0


# ---- GPU: zeros and infinities ------------------------------------------------------------------

@gpu
@pytest.mark.parametrize("kernel", [api.KERNEL_SIMPLE, api.KERNEL_TILED])
@pytest.mark.parametrize("name", STARS)
def test_positive_zero_regions_and_infinite_walls(name, kernel):
    reach = int(np.abs(W.star(name)).max())
    dims = (16 + 2 * reach,) * 3 if reach < 7 else (36, 34, 32)
    v = W.random_field(dims, seed=3)
    v[:, :, :4] = 0.0  # +0.0 floor
    lo = tuple((n - 6) // 2 - reach for n in dims)
    hi = tuple(a + 6 + 2 * reach for a in lo)
    v[lo[0]:hi[0], lo[1]:hi[1], lo[2]:hi[2]] = np.inf  # a wall as thick as the star's reach...
    pocket = tuple(slice(a + reach, b - reach) for a, b in zip(lo, hi))
    v[pocket] = 0.2  # ... around a pocket no edge can enter
    starts = [(1, 1, 1), (dims[0] - 1, 2, 0), (0, dims[1] - 1, dims[2] - 1)]
    tts, _ = _check_against_oracle(v, name, starts, kernel=kernel, what=f"{name}-FS walls")
    for tt in tts:
        assert np.isinf(tt[pocket]).all() and np.isfinite(tt[:, :, :4]).all()


@gpu
@pytest.mark.parametrize("name", STARS)
def test_infinite_start_and_an_infinite_model(name):
    v = W.random_field(DIMS, seed=5)
    start = (5, 6, 7)
    v[start] = np.inf
    tts, _ = _check_against_oracle(v, name, [start], what="infinite start")
    want = np.full(DIMS, np.inf, F)
    want[start] = 0
    assert_bit_equal(tts[0], want, "infinite start")
    v = np.full(DIMS, np.inf, F)
    v[start] = 0.3
    tts, _ = _check_against_oracle(v, name, [start, (0, 0, 0)], what="infinite model")
    assert_bit_equal(tts[0], want, "infinite model")


# ---- GPU: delta ---------------------------------------------------------------------------------

@gpu
@pytest.mark.parametrize("delta", [1.0, 0.1, 0.3, 2.5, 1e-3, 1e3, 1e-20, 1e20])
@pytest.mark.parametrize("name", STARS)
def test_non_default_delta(name, delta):
    v = W.random_field((20, 18, 16), seed=11)
    starts = [(3, 4, 5), (19, 0, 15)]
    assert guard_accepts(*star_range(W.star(name), delta), *model_range(v))
    for kernel in (api.KERNEL_SIMPLE, api.KERNEL_TILED):
        _check_against_oracle(v, name, starts, delta=delta, kernel=kernel, what=f"delta {delta} kernel {kernel}")


@gpu
def test_non_default_delta_one_shot_and_over_slabs():
    v = W.random_field((22, 18, 16), seed=12)
    off, start = W.star("818"), (3, 4, 5)
    for delta in (0.3, 1e-20):
        ref, _, _ = oracle.solve(v, off, start, delta=delta)
        tt, _ = P.solve(v, off, [start], delta=delta)
        assert_bit_equal(tt[0], ref, f"sweeptt_solve, delta {delta}")
        tt, _ = P.solve_slabs(v, off, start, num_slabs=2, slab_axis=0, delta=delta)
        assert_bit_equal(tt, ref, f"sweeptt_solve_slabs, delta {delta}")
    P.load_library().sweeptt_release_cache()


# ---- GPU: dynamic range inside the domain --------------------------------------------------------

@gpu
@pytest.mark.parametrize("name", ["3", "818"])
def test_slowness_over_sixty_decades(name):
    rng = np.random.default_rng(13)
    v = (10.0 ** rng.uniform(-30, 30, size=(22, 20, 18))).astype(F)
    for kernel in (api.KERNEL_SIMPLE, api.KERNEL_TILED):
        _check_against_oracle(v, name, [(3, 4, 5), (21, 19, 0)], kernel=kernel, what=f"log-uniform, kernel {kernel}")


@gpu
@pytest.mark.parametrize("name", ["3", "818"])
def test_travel_times_that_overflow_on_both_sides(name):
    v = np.full((40, 12, 10), 1e36, F)
    assert guard_accepts(*star_range(W.star(name), 10.0), *model_range(v))
    tts, _ = _check_against_oracle(v, name, [(0, 5, 5)], what="constant 1e36")
    assert np.isinf(tts[0]).any() and np.isfinite(tts[0]).sum() > 1


def _bound_model(name, delta=10.0):
    """A model with the last accepted vmax and the first accepted vpos of the star at delta."""
    dmax, dpos = star_range(W.star(name), delta)
    v = W.random_field((20, 18, 16), seed=14)
    top, bottom = last_vmax(dmax), first_vpos(dpos)
    v[10:12, 2:5, 3] = top
    v[4, 10:14, 8:10] = bottom
    return v, top, bottom


@gpu
@pytest.mark.parametrize("name", STARS)
def test_models_on_the_last_accepted_float_of_each_bound(name):
    v, top, bottom = _bound_model(name)
    assert model_range(v) == (top, bottom)
    for kernel in (api.KERNEL_SIMPLE, api.KERNEL_TILED):
        _check_against_oracle(v, name, [(3, 4, 5), (11, 3, 3), (4, 11, 9)], kernel=kernel, what=f"bounds {kernel}")


@gpu
def test_distance_on_the_bound_is_accepted():
    v = (W.random_field((20, 18, 16), seed=15) * 10).astype(F)  # slowness >= 1: dpos * vpos >= 2^-125 with dpos = 2^-125
    delta = float(LO)
    assert star_range(W.star("3"), delta)[1] == LO and guard_accepts(*star_range(W.star("3"), delta), *model_range(v))
    _check_against_oracle(v, "3", [(3, 4, 5)], delta=delta, what="d = 2^-125")


# ---- GPU: refusals ------------------------------------------------------------------------------

def _beyond_models(name):
    """(what, model, delta, message) one float beyond each bound."""
    v, top, bottom = _bound_model(name)
    over = v.copy()
    over[10, 2, 3] = np.nextafter(top, F(np.inf))
    under = v.copy()
    under[4, 10, 8] = np.nextafter(bottom, F(0))
    small_d = (W.random_field((20, 18, 16), seed=15) * 10).astype(F)
    return [("vmax", over, 10.0, "overflows"), ("vpos", under, 10.0, r"below 2\^-125"),
            ("d", small_d, float(np.nextafter(LO, F(0))), r"below 2\^-125")]


@gpu
@pytest.mark.parametrize("name", ["3", "818"])
def test_models_beyond_each_bound_are_refused_everywhere(name):
    start = (3, 4, 5)
    for what, v, delta, msg in _beyond_models(name):
        assert not guard_accepts(*star_range(W.star(name), delta), *model_range(v)), what
        with P.SweepContext() as ctx:
            ctx.set_model(v); ctx.set_star(W.star(name), delta); ctx.set_sources([start])
            for call in (ctx.run, ctx.step, ctx.reset, lambda: ctx.trace_rays([start]),
                         lambda: ctx.freeze_rays([start])):
                with pytest.raises(P.SweepError, match=msg):
                    call()
        with pytest.raises(P.SweepError, match=msg):
            P.solve(v, W.star(name), [start], delta=delta)
        with pytest.raises(P.SweepError, match=msg):
            P.solve_slabs(v, W.star(name), start, num_slabs=2, slab_axis=0, delta=delta)
    P.load_library().sweeptt_release_cache()


def _bad_stars():
    off = W.star("5")
    hand = P.make_star(off, 10.0)
    hand[7].d = -hand[7].d
    return [("delta -10", P.make_star(off, -10.0)), ("delta nan", P.make_star(off, float("nan"))),
            ("delta inf", P.make_star(off, float("inf"))), ("one negative d", hand)]


@gpu
def test_stars_with_negative_nan_or_infinite_distances_are_refused():
    v = W.random_field((20, 18, 16), seed=16)
    for what, fs in _bad_stars():
        with P.SweepContext() as ctx:
            ctx.set_model(v)
            with pytest.raises(P.SweepError, match="finite d >= 0"):
                ctx.set_star(fs)
            with pytest.raises(P.SweepError, match="a model, a star"):
                ctx.set_sources([(1, 2, 3)]); ctx.run()
        with pytest.raises(P.SweepError, match="finite d >= 0"):
            P.solve(v, fs, [(1, 2, 3)])
    P.load_library().sweeptt_release_cache()


@gpu
@pytest.mark.parametrize("kernel", [api.KERNEL_SIMPLE, api.KERNEL_TILED])
def test_refused_calls_leave_the_context_as_it_was(kernel):
    v = W.random_field((20, 18, 16), seed=17)
    off, starts = W.star("5"), [(3, 4, 5), (19, 0, 15)]
    refs = [oracle.solve(v, off, p)[0] for p in starts]
    neg = v.copy(); neg[5, 5, 5] = -0.1
    nan = v.copy(); nan[1, 2, 3] = np.nan
    wide = np.concatenate([off[:-1], [[9, 1, 0], [0, 0, 0]]]).astype(np.int32)  # |i| = 9: beyond the tiled halo
    refused = [("negative model", lambda c: c.set_model(neg), "negative or NaN"),
               ("NaN model of other dimensions", lambda c: c.set_model(W.random_field((9, 30, 7)) * np.nan),
                "negative or NaN"),
               ("NaN model", lambda c: c.set_model(nan), "negative or NaN"),
               ("no usable offsets", lambda c: c.set_star(np.zeros((3, 3), np.int32)), "no usable offsets")]
    refused += [(what, lambda c, fs=fs: c.set_star(fs), "finite d >= 0") for what, fs in _bad_stars()]
    if kernel == api.KERNEL_TILED:
        refused.append(("star beyond the tiled halo", lambda c: c.set_star(wide), "tiled kernel holds"))
    mark = np.full(v.shape, 7.0, F)
    with P.SweepContext(kernel=kernel) as ctx:
        ctx.set_model(v); ctx.set_star(off); ctx.set_sources(starts)
        ctx.run()
        stats = ctx.model_stats()
        for what, call, msg in refused:
            ctx.put_tt(0, mark)
            with pytest.raises(P.SweepError, match=msg):
                call(ctx)
            # right after the refusal: same dimensions, sources, statistics and travel-time boxes
            assert ctx.dims == v.shape and ctx.nsrc == len(starts) and ctx.model_stats() == stats, what
            assert_bit_equal(ctx.get_tt(0), mark, f"box 0 right after the refused {what}")
            assert_bit_equal(ctx.get_tt(1), refs[1], f"box 1 right after the refused {what}")
            ctx.reset()
            ctx.run()
            for s in range(len(starts)):
                assert_bit_equal(ctx.get_tt(s), refs[s], f"after the refused {what}, source {s}")
                assert ctx.count_violations(s) == 0, what


@gpu
def test_a_model_whose_axis_order_the_star_cannot_follow_is_refused_whole():
    """The tiled kernel holds |k| <= 8 but only |i| <= 7.  A star with (0, 0, +-8) fits while the caller's z is the
    kernel's z (16^3: the caller's order); a 16 x 16 x 12 model puts the caller's z on the kernel's x (12 fills whole
    4-wide units, not whole 8-deep tiles), where the star does not fit.  That model is refused before anything
    changes: the previous model, star and sources still solve bit for bit."""
    off = np.concatenate([W.star("5")[:-1], [[0, 0, 8], [0, 0, 0]]]).astype(np.int32)
    v = W.random_field((16, 16, 16), seed=18)
    starts = [(3, 4, 5), (15, 0, 15)]
    refs = [oracle.solve(v, off, p)[0] for p in starts]
    mark = np.full(v.shape, 7.0, F)
    with P.SweepContext(kernel=api.KERNEL_TILED) as ctx:
        ctx.set_model(v); ctx.set_star(off); ctx.set_sources(starts)
        ctx.run()
        stats = ctx.model_stats()
        ctx.put_tt(0, mark)
        with pytest.raises(P.SweepError, match="tiled kernel holds"):
            ctx.set_model(W.random_field((16, 16, 12), seed=19))
        assert ctx.dims == v.shape and ctx.nsrc == 2 and ctx.model_stats() == stats
        assert_bit_equal(ctx.get_tt(0), mark, "box 0 right after the refused model")
        assert_bit_equal(ctx.get_tt(1), refs[1], "box 1 right after the refused model")
        ctx.run()
        for s in range(2):
            assert_bit_equal(ctx.get_tt(s), refs[s], f"source {s} after the refused model")
            assert ctx.count_violations(s) == 0
    with P.SweepContext() as ctx:  # the automatic choice takes the simple kernel for that model instead
        w = W.random_field((16, 16, 12), seed=19)
        ctx.set_model(w); ctx.set_star(off); ctx.set_sources(starts[:1])
        assert ctx.run().kernel_used == api.KERNEL_SIMPLE
        assert_bit_equal(ctx.get_tt(0), oracle.solve(w, off, starts[0])[0], "simple kernel, 16 x 16 x 12")


@gpu
def test_model_statistics_fold_negative_zero():
    """The exact minimum feeds the downwind filter's lower bound dmin = hd_min * 2 vmin: with -0.0 in the model it
    must be 0, not the smallest positive value (-0.0's bits order above every positive float)."""
    cases = [(v, what) for what, (v, _) in _signed_zero_models().items()]
    cases += [(_twin(v), what + " +0.0") for v, what in list(cases)]
    v = W.random_field(DIMS, seed=20)
    cases += [(v, "positive"), (_bound_model("818")[0], "bounds")]
    inf = np.full(DIMS, np.inf, F); inf[1, 2, 3] = -0.0
    cases += [(inf, "+INF and one -0.0"), (np.full(DIMS, np.inf, F), "+INF only")]
    with P.SweepContext() as ctx:
        for v, what in cases:
            ctx.set_model(v)
            fin = v[np.isfinite(v)]
            want_min = F(np.abs(fin).min()) if len(fin) else F(-1)
            got = ctx.model_stats()
            assert got[0].view(np.uint32) == want_min.view(np.uint32), (what, got, want_min)
            assert (got[1], got[2]) == model_range(v), (what, got)
