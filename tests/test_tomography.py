"""Tomography operators over the rays (include/sweeptt.h, sweeptt_ray_project / sweeptt_ray_backproject).

The oracle is the ray oracle of test_rays.py plus exact arithmetic here: the projection replays the contract's float
expression in numpy float32 from the start end, the back-projection sums the integer quanta rint_even(w*hd*2^-E) in
int64 and rounds each node's sum once to float32 with Python integers.  CPU: the oracle projection of the slowness is
the field itself on every golden node; G and G^T are adjoint up to a bound derived from the float32 path sums; a ray's
row of G is a supergradient of its travel time (CPU sweep oracle); the new kernels never fuse a multiply-add; a C99
client links.  GPU (-m gpu): device results equal the oracle bit for bit on every golden node whatever kernel, axis
permutation or put_tt produced the field; rays that are not OK contribute nothing; truncation and the default retry;
determinism; source slicing; full-size config 2; misfit_gradient."""
import hashlib
import json
import math
import re
import shutil
import subprocess
from fractions import Fraction

import numpy as np
import pytest
import torch

import oracle
import uoparallel_seismic_project_b200 as P
from uoparallel_seismic_project_b200 import api, workloads as W

from conftest import ROOT, make_field
from test_rays import _golden_cases, _oracle_rays, all_nodes, half_distance, oracle_rays

gpu = pytest.mark.gpu
OK, TRUNCATED = api.RAY_OK, api.RAY_TRUNCATED
U = 2.0 ** -24   # unit roundoff of float32


# ---- oracle ------------------------------------------------------------------------------------

def _edges(nodes, length):
    """Per ray, its edges from the START end: yields (live[R], n[R,3], m[R,3]) with n nearer the receiver."""
    nodes = nodes.astype(np.int64)
    R, L = nodes.shape[:2]
    rows = np.arange(R)
    last = length.astype(np.int64) - 1
    for back in range(1, int(length.max(initial=1))):
        live = last - back >= 0
        k = np.where(live, last - back, 0)
        yield live, nodes[rows, k], nodes[rows, np.minimum(k + 1, L - 1)]


def oracle_project(d, nodes, length, status, delta=10.0):
    """acc = +0; for each edge (n, m) from the start end: acc = fl(fl(hd * fl(d_n + d_m)) + acc).  NaN unless OK."""
    d = np.asarray(d, np.float32)
    acc = np.zeros(len(length), np.float32)
    for live, n, m in _edges(nodes, length):
        with np.errstate(over="ignore", invalid="ignore"):
            term = half_distance(m - n, delta) * (d[tuple(n.T)] + d[tuple(m.T)])
            acc = np.where(live, term + acc, acc).astype(np.float32)
    return np.where(status == OK, acc, np.float32(np.nan)).astype(np.float32)


def quantum_exp(hd_max, wmax, n):
    """Smallest E with 2*hd_max*W*N <= 2^(E+62), in exact rationals (0 when W or hd_max is 0)."""
    if wmax == 0 or hd_max == 0:
        return 0
    f = Fraction(2) * Fraction(float(hd_max)) * Fraction(float(wmax)) * n
    e = f.numerator.bit_length() - f.denominator.bit_length() - 62
    while f > Fraction(2) ** (e + 62):
        e += 1
    while f <= Fraction(2) ** (e + 61):
        e -= 1
    return e


def _quanta(w, hd, e):
    """rint_even(w * hd * 2^-e) as int64, from the integer significands (no floating point)."""
    mw, ew = np.frexp(w.astype(np.float64))
    mh, eh = np.frexp(hd.astype(np.float64))
    x = np.abs(np.rint(mw * 2.0 ** 24).astype(np.int64) * np.rint(mh * 2.0 ** 24).astype(np.int64))  # < 2^48
    s = (ew + eh - 48 - e).astype(np.int64)   # |w * hd * 2^-e| = x * 2^s
    out = np.zeros_like(x)
    up = s >= 0
    out[up] = x[up] << s[up]
    sh = np.minimum(-s, 62)
    dn = ~up
    q = x[dn] >> sh[dn]
    rem = x[dn] - (q << sh[dn])
    half = np.int64(1) << (sh[dn] - 1)
    q += (rem > half) | ((rem == half) & (q & 1 == 1))
    out[dn] = q
    return np.where(w < 0, -out, out)


def round_once(total, e):
    """float32 nearest (ties to even) of the integer `total` times 2^e, subnormals and overflow included."""
    if total == 0:
        return np.float32(0.0)
    u = abs(int(total))
    top = u.bit_length() - 1 + e          # 2^top <= |value| < 2^(top+1)
    qe = max(top - 23, -149)              # quantum of the float32 binade (or of the subnormals)
    sh = qe - e
    if sh <= 0:
        r = u << -sh
    else:
        r, rem = u >> sh, u & ((1 << sh) - 1)
        if rem > (1 << (sh - 1)) or (rem == (1 << (sh - 1)) and r & 1):
            r += 1
    mag = np.float32(np.inf) if r * Fraction(2) ** qe >= Fraction(2) ** 128 else np.float32(math.ldexp(r, qe))
    return -mag if total < 0 else mag


def oracle_backproject(dims, rays, weights, hd_max, delta=10.0):
    """rays: list over sources of (nodes, length, status); weights [S, R].  Returns (grad float32[dims], E)."""
    w = np.asarray(weights, np.float32)
    e = quantum_exp(hd_max, float(np.abs(w).max(initial=0)), w.size)
    acc = np.zeros(int(np.prod(dims)), np.int64)
    for (nodes, length, status), ws in zip(rays, w):
        use = (status == OK) & (ws != 0)
        for live, n, m in _edges(nodes[use], length[use]):
            c = _quanta(ws[use][live], half_distance(m[live] - n[live], delta), e)
            np.add.at(acc, np.ravel_multi_index(tuple(n[live].T), dims), c)
            np.add.at(acc, np.ravel_multi_index(tuple(m[live].T), dims), c)
    grad = np.zeros(acc.shape, np.float32)
    for j in np.nonzero(acc)[0]:
        grad[j] = round_once(int(acc[j]), e)
    return grad.reshape(dims), e


def _hd_max(star, delta=10.0):
    off = np.asarray(W.star(star) if isinstance(star, str) else star)[:-1]
    return float(half_distance(off[np.abs(off).sum(1) > 0], delta).max())


def _weights(shape, seed):
    """Signs mixed, about a tenth zeros, magnitudes over 40 binades."""
    rng = np.random.default_rng(seed)
    w = (rng.uniform(0.5, 1.0, shape) * 2.0 ** rng.integers(-20, 21, shape) * rng.choice([-1, 1], shape))
    w[rng.random(shape) < 0.1] = 0
    return w.astype(np.float32)


# ---- CPU: the oracle ---------------------------------------------------------------------------

def test_oracle_projection_of_the_slowness_is_the_field():
    for case, ms in _golden_cases().items():
        v = make_field(ms[0]["kind"], ms[0]["dims"], ms[0]["seed"])
        for m, (nodes, length, status, _) in zip(ms, _oracle_rays(case)):
            got = oracle_project(v, nodes, length, status)
            want = m["tt"].ravel()
            nd = int((got.view(np.uint32) != want.view(np.uint32)).sum())
            assert nd == 0, f"{case}[{m['idx']}]: {nd} of {len(want)} nodes differ"


def test_round_once_matches_numpy_where_a_double_is_exact():
    rng = np.random.default_rng(5)
    for _ in range(2000):
        total = int(rng.integers(-(1 << 52), 1 << 52))
        e = int(rng.integers(-200, 90))
        want = np.float32(math.ldexp(total, e)) if abs(math.ldexp(total, e)) < 3.4e38 else None
        if want is not None and np.isfinite(want) and abs(math.ldexp(total, e)) >= 2.0 ** -126:
            got = round_once(total, e)   # one rounding from an exact double is the float32 rounding (normal range)
            assert got.view(np.uint32) == want.view(np.uint32), (total, e)
    assert round_once(3, -150).view(np.uint32) == 2          # 1.5 quanta -> 2 (ties to even)
    assert round_once(1, -150).view(np.uint32) == 0          # 0.5 quantum -> 0
    assert round_once(-1, -150).view(np.uint32) == 0x80000000
    assert round_once((1 << 24) - 1, -150).view(np.uint32) == 0x00800000   # rounds up to the smallest normal
    assert np.isinf(round_once(1, 128)) and round_once((1 << 24) - 1, 104) == np.float32(3.4028235e38)


def test_quantum_exponent_is_the_smallest():
    for hd, wm, n in [(5.0, 1.0, 1), (7.0710678, 3.5e-20, 58081 * 4), (1e-30, 1e30, 3), (0.5, 2.0 ** -149, 1)]:
        e = quantum_exp(np.float32(hd), np.float32(wm), n)
        f = Fraction(2) * Fraction(float(np.float32(hd))) * Fraction(float(np.float32(wm))) * n
        assert f <= Fraction(2) ** (e + 62) and f > Fraction(2) ** (e + 61)


def _case_rays(case):
    return [(nodes, length, status) for nodes, length, status, _ in _oracle_rays(case)]


@pytest.mark.parametrize("case", ["rand_818", "contrast_5fs", "hetero_818"])
def test_oracle_operators_are_adjoint(case):
    """<G x, w> = <x, G^T w> up to the rounding of both sides.  G x: each term hd*(x_n + x_m) and each of the L-1
    additions of a ray's float32 sum round once, so |err_q| <= (L_q + 1) u sum_e hd_e (|x_n| + |x_m|) (to first order;
    the bound is taken 1% wider).  G^T w: every contribution is off by at most half a quantum 2^(E-1), and every node's
    sum is rounded once more (u |g_j|).  The float64 dot products add a relative 1e-12."""
    ms = _golden_cases()[case]
    dims = tuple(ms[0]["dims"])
    rays = _case_rays(case)
    rng = np.random.default_rng(11)
    x = rng.standard_normal(dims).astype(np.float32)
    w = _weights((len(ms), int(np.prod(dims))), 3)
    gx = [oracle_project(x, *r) for r in rays]
    g, e = oracle_backproject(dims, rays, w, _hd_max(ms[0]["star"]))
    lhs = sum(float(np.dot(a.astype(np.float64), b.astype(np.float64))) for a, b in zip(gx, w))
    rhs = float(np.dot(x.ravel().astype(np.float64), g.ravel().astype(np.float64)))
    bound = 0.0
    counts = np.zeros(int(np.prod(dims)), np.float64)
    ax = np.abs(x.astype(np.float64))
    for (nodes, length, status), ws in zip(rays, w):
        mag = np.zeros(len(length))
        for live, n, m in _edges(nodes, length):
            hd = half_distance(m - n).astype(np.float64)
            mag += np.where(live, hd * (ax[tuple(n.T)] + ax[tuple(m.T)]), 0)
            np.add.at(counts, np.ravel_multi_index(tuple(n[live].T), dims), 1)
            np.add.at(counts, np.ravel_multi_index(tuple(m[live].T), dims), 1)
        bound += 1.01 * float(np.sum(np.abs(ws) * (length + 1) * U * mag))
    bound += float(np.sum(ax.ravel() * (counts * 2.0 ** (e - 1) + U * np.abs(g.ravel()))))
    bound += 1e-12 * (abs(lhs) + abs(rhs))
    assert abs(lhs - rhs) <= bound, (lhs, rhs, bound)
    assert abs(lhs - rhs) > 0 or bound > 0


def test_ray_row_is_a_supergradient_of_the_travel_time():
    """T is a minimum over paths of sums linear in the slowness, so T(v + h) <= T(v) + G h.  Checked with the CPU sweep
    oracle for h = +-eps e_j at sampled (ray, node j) pairs, j on the ray or next to it.  Slack: both travel times are
    float32 sums along paths of at most L edges, each step rounding twice, so each is within 2 L u T of its exact value
    (taken 2x wider)."""
    ms = _golden_cases()["rand_5fs"]
    m = ms[0]
    v = make_field(m["kind"], m["dims"], m["seed"])
    star = W.star(m["star"])
    start = tuple(m["start"])
    nodes, length, status, _ = oracle_rays(v, m["tt"], star, start, all_nodes(v.shape))
    rng = np.random.default_rng(9)
    picks = rng.choice(np.nonzero(length >= 4)[0], 6, replace=False)
    checked = 0
    for r in picks:
        path = nodes[r, : length[r]]
        row = np.zeros(v.shape, np.float64)   # G[r, :] in float64: sum of hd over the edges touching each node
        for a, b in zip(path[:-1], path[1:]):
            hd = float(half_distance((b - a)[None])[0])
            row[tuple(a)] += hd
            row[tuple(b)] += hd
        rec = tuple(path[0])
        t0 = float(m["tt"][rec])
        for j in [tuple(path[len(path) // 2]), tuple(path[1]), tuple(np.minimum(path[1] + 1, np.array(v.shape) - 1))]:
            for sgn in (1, -1):
                eps = 0.25 * float(v[j]) * sgn
                vp = v.copy()
                vp[j] = np.float32(v[j] + eps)
                h = float(vp[j]) - float(v[j])
                tp, _, _ = oracle.solve(vp, star, start)
                slack = 4 * length[r] * U * (t0 + abs(float(tp[rec])))
                assert float(tp[rec]) <= t0 + h * row[j] + slack, (rec, j, sgn, float(tp[rec]), t0, h * row[j])
                checked += 1
    assert checked == 36


# ---- CPU: the shipped library ------------------------------------------------------------------

@pytest.mark.skipif(shutil.which("cuobjdump") is None, reason="cuobjdump not on PATH")
def test_tomography_kernels_never_fuse_multiply_add():
    out = subprocess.run(["cuobjdump", "-sass", str(P.lib_path())], capture_output=True, text=True, check=True).stdout
    funcs, name = {}, None
    for line in out.splitlines():
        mm = re.search(r"Function : (\S+)", line)
        if mm:
            name = mm.group(1)
            funcs[name] = []
        elif name and re.match(r"\s+/\*[0-9a-f]{4,6}\*/", line):
            funcs[name].append(line)
    kernels = {k: v for k, v in funcs.items() if re.search("ray_project|ray_backproject|grad_finish", k)}
    assert len(kernels) == 3, sorted(kernels)
    for k, lines in kernels.items():
        text = "\n".join(lines)
        if "ray_project" in k:
            assert "FMUL" in text and "FADD" in text, k
        assert not re.search(r"\bFFMA2?\b", text), f"{k}: fused multiply-add found"


def test_c99_client_calls_the_tomography_operators(tmp_path):
    """A strict C99 client compiles and links against both entry points.  Without a GPU each fails with a message;
    with one, a tiny constant box: the projection of the slowness is the receiver's time and the coverage of the
    straight ray is hd at its ends and 2 hd inside."""
    src = tmp_path / "client.c"
    src.write_text(r'''
#include <stdio.h>
#include "sweeptt.h"
int main(void) {
  struct FS fs[7] = {{1, 0, 0, 0.f}, {-1, 0, 0, 0.f}, {0, 1, 0, 0.f}, {0, -1, 0, 0.f}, {0, 0, 1, 0.f},
                     {0, 0, -1, 0.f}, {1, 1, 1, 0.f}};
  struct START st[1] = {{0, 0, 0}}, rec[2] = {{3, 0, 0}, {0, 0, 0}};
  float v[64], proj[2], w[2] = {1.f, 1.f}, grad[64];
  int32_t len[2], status[2];
  int e = -1, i;
  sweeptt_stats stats;
  sweeptt_ctx *ctx;
  for (i = 0; i < 64; i++) v[i] = 1.f;
  sweeptt_star_fill_distances(fs, 7, 10.0f);
  ctx = sweeptt_create(NULL);
  if (!ctx) {
    if (sweeptt_ray_project(NULL, 0, 1, rec, 2, 16, v, proj, status, len, &stats)) return 2;
    printf("%s\n", sweeptt_last_error());
    if (sweeptt_ray_backproject(NULL, 0, 1, rec, 2, 16, w, grad, &e, status, &stats)) return 2;
    printf("%s\n", sweeptt_last_error());
    return 0;
  }
  if (!sweeptt_set_model(ctx, v, 4, 4, 4) || !sweeptt_set_star(ctx, fs, 7) || !sweeptt_set_sources(ctx, st, 1) ||
      !sweeptt_run(ctx, NULL) || !sweeptt_ray_project(ctx, 0, 1, rec, 2, 16, v, proj, status, len, &stats) ||
      !sweeptt_ray_backproject(ctx, 0, 1, rec, 2, 16, w, grad, &e, status, &stats)) {
    printf("%s\n", sweeptt_last_error());
    return 3;
  }
  sweeptt_destroy(ctx);
  if (status[0] != SWEEPTT_RAY_OK || len[0] != 4 || proj[0] != 30.f || proj[1] != 0.f) return 4;
  if (grad[0] != 5.f || grad[16] != 10.f || grad[32] != 10.f || grad[48] != 5.f || grad[1] != 0.f) return 5;
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

def _ctx(ms, kernel=None, put=False):
    v = make_field(ms[0]["kind"], ms[0]["dims"], ms[0]["seed"])
    ctx = P.SweepContext(kernel=kernel)
    ctx.set_model(v); ctx.set_star(W.star(ms[0]["star"])); ctx.set_sources([m["start"] for m in ms])
    if put:
        for s, m in enumerate(ms):
            ctx.put_tt(s, m["tt"])
    else:
        ctx.run()
    return ctx, v


def _bits_equal(a, b):
    return np.array_equal(np.asarray(a, np.float32).view(np.uint32), np.asarray(b, np.float32).view(np.uint32))


def _check_every_golden(**kw):
    for case, ms in _golden_cases().items():
        dims = tuple(ms[0]["dims"])
        rec = all_nodes(dims)
        rays = _oracle_rays(case)
        ctx, v = _ctx(ms, **kw)
        with ctx:
            d = np.random.default_rng(1).standard_normal(dims).astype(np.float32)
            w = _weights((len(ms), len(rec)), 2)
            pv = ctx.ray_project(v, rec)
            pd = ctx.ray_project(d, rec)
            bp = ctx.ray_backproject(w, rec)
        assert pd.stats.kernel_launches == 2 and pd.stats.relaxations > 0 and pd.stats.solve_ms > 0
        assert bp.stats.kernel_launches == 2 and bp.stats.relaxations > 0 and bp.stats.solve_ms > 0
        for s, (m, (nodes, length, status, _)) in enumerate(zip(ms, rays)):
            what = f"{case}[{s}] {kw}"
            assert (pd.status[s] == status).all() and (pd.length[s] == length).all(), what
            assert (bp.status[s] == status).all(), what
            assert _bits_equal(pv.values[s], m["tt"].ravel()), f"{what}: projection of the slowness != tt"
            assert _bits_equal(pd.values[s], oracle_project(d, nodes, length, status)), f"{what}: projection"
        g, e = oracle_backproject(dims, [r[:3] for r in rays], w, _hd_max(ms[0]["star"]))
        assert bp.quantum_exp == e, (case, bp.quantum_exp, e)
        assert _bits_equal(bp.grad, g), f"{case} {kw}: back-projection differs in {int((bp.grad != g).sum())} nodes"


@gpu
@pytest.mark.parametrize("kernel", [api.KERNEL_SIMPLE, api.KERNEL_TILED])
def test_device_operators_equal_oracle_on_every_golden_node(kernel):
    _check_every_golden(kernel=kernel)


@gpu
@pytest.mark.parametrize("axis", ["0", "1", "2"])
def test_device_operators_do_not_depend_on_the_axis_permutation(axis, monkeypatch):
    monkeypatch.setenv("SWEEPTT_WINDOW_AXIS", axis)
    _check_every_golden()


@gpu
def test_device_operators_of_fields_loaded_with_put_tt():
    _check_every_golden(put=True)


def _assert_not_ok_rays_contribute_nothing(ctx, v, dims, what):
    rec = all_nodes(dims)
    rng = np.random.default_rng(4)   # W = 1 whichever rays are OK, so the quantum is the same with or without them
    w = rng.choice(np.array([1.0, -1.0, 0.5], np.float32), (ctx.nsrc, len(rec)))
    pr = ctx.ray_project(v, rec)
    bp = ctx.ray_backproject(w, rec)
    assert (pr.status != OK).any(), f"{what}: every ray is OK"
    assert np.isnan(pr.values[pr.status != OK]).all() and not np.isnan(pr.values[pr.status == OK]).any(), what
    # only the OK rays: the same result with the weights of every other ray set to 0
    w_ok = np.where(bp.status == OK, w, np.float32(0))
    ref = ctx.ray_backproject(w_ok, rec)
    assert (ref.status == bp.status).all() and ref.quantum_exp == bp.quantum_exp
    assert _bits_equal(bp.grad, ref.grad), what


@gpu
def test_rays_that_are_not_ok_contribute_nothing():
    ms = _golden_cases()["hetero_818"]
    dims = tuple(ms[0]["dims"])
    ctx, v = _ctx(ms, put=True)
    with ctx:
        ctx.reset()
        ctx.step(3)   # not converged: some rays are NOT_FIXED_POINT / NO_PREDECESSOR
        _assert_not_ok_rays_contribute_nothing(ctx, v, dims, "unconverged")
    ms = _golden_cases()["rand_818"]
    dims = tuple(ms[0]["dims"])
    ctx, v = _ctx(ms, put=True)
    with ctx:
        bad = ms[0]["tt"].copy()
        bad[tuple(np.array(dims) // 2)] *= np.float32(0.5)   # inconsistent field
        ctx.put_tt(0, bad)
        _assert_not_ok_rays_contribute_nothing(ctx, v, dims, "inconsistent put_tt")


@gpu
def test_small_max_nodes_truncates():
    ms = _golden_cases()["hetero_818"]
    dims = tuple(ms[0]["dims"])
    rec = all_nodes(dims)[::5]
    w = np.ones((len(ms), len(rec)), np.float32)
    ctx, v = _ctx(ms)
    with ctx:
        short = ctx.ray_project(v, rec, max_nodes=3)
        short_bp = ctx.ray_backproject(w, rec, max_nodes=3)
        with pytest.raises(P.SweepError, match="max_nodes"):
            ctx.ray_project(v, rec, max_nodes=0)
        with pytest.raises(P.SweepError, match="not finite"):
            ctx.ray_backproject(np.full_like(w, np.nan), rec)
        with pytest.raises(P.SweepError, match="outside"):
            ctx.ray_backproject(w[:, :1], [(0, 0, 99)])
    assert (short.status == TRUNCATED).any() and (short.status == OK).any() and (short.length <= 3).all()
    assert np.isnan(short.values[short.status == TRUNCATED]).all()
    assert (short_bp.status == short.status).all()


# the six axis neighbours (symmetric, so that the nodes next to the start can pull from it; the last row is not used)
AXIS_STAR = np.array([[1, 0, 0], [-1, 0, 0], [0, 1, 0], [0, -1, 0], [0, 0, 1], [0, 0, -1], [0, 0, 0]], np.int32)


def _maze():
    """A 9 x 9 x 1 model whose walls (x = 1, 3, 5, 7; +INF slowness) leave a gap at alternating ends: with axis steps
    only, the ray from the far corner winds through every corridor, far longer than nx+ny+nz = 19 nodes."""
    v = np.ones((9, 9, 1), np.float32)
    for i, x in enumerate((1, 3, 5, 7)):
        v[x, :, 0] = np.inf
        v[x, 8 if i % 2 == 0 else 0, 0] = 1.0
    return v


@gpu
def test_default_max_nodes_grows_until_no_ray_is_truncated():
    v = _maze()
    star = AXIS_STAR
    start, far = (0, 0, 0), (8, 8, 0)
    tt, _, _ = oracle.solve(v, star, start)
    nodes, length, status, _ = oracle_rays(v, tt, star, start, [far], max_nodes=200)
    assert status[0] == OK and length[0] > 2 * sum(v.shape), length[0]
    with P.SweepContext() as ctx:
        ctx.set_model(v); ctx.set_star(star); ctx.set_sources([start])
        ctx.run()
        cut = ctx.ray_project(v, [far], max_nodes=sum(v.shape))
        grown = ctx.ray_project(v, [far])
        cov = ctx.ray_backproject(np.ones((1, 1), np.float32), [far])
    assert cut.status[0, 0] == TRUNCATED
    assert grown.status[0, 0] == OK and grown.length[0, 0] == length[0]
    assert _bits_equal(grown.values[0, 0], tt[far]) and cov.status[0, 0] == OK
    want, e = oracle_backproject(v.shape, [(nodes, length, status)], np.ones((1, 1), np.float32), _hd_max(AXIS_STAR))
    assert cov.quantum_exp == e and _bits_equal(cov.grad, want)


@gpu
def test_back_projection_is_deterministic():
    ms = _golden_cases()["hetero_818"]
    dims = tuple(ms[0]["dims"])
    rec = all_nodes(dims)
    w = _weights((len(ms), len(rec)), 8)
    ctx, v = _ctx(ms)
    with ctx:
        a = ctx.ray_backproject(w, rec)
        b = ctx.ray_backproject(w, rec)
    assert a.quantum_exp == b.quantum_exp and _bits_equal(a.grad, b.grad)


@gpu
def test_path_records_in_global_memory_give_the_same_results():
    """With max_nodes = 20,000 the eight per-warp path records (320 KB) cannot sit in shared memory next to the pull
    table, so they go to a global slot per resident warp; the results are those of the default call."""
    ms = _golden_cases()["hetero_818"]
    dims = tuple(ms[0]["dims"])
    rec = all_nodes(dims)[::3]
    d = np.random.default_rng(12).standard_normal(dims).astype(np.float32)
    w = _weights((len(ms), len(rec)), 13)
    ctx, v = _ctx(ms)
    with ctx:
        pool = ctx.pool_bytes
        p_small, b_small = ctx.ray_project(d, rec), ctx.ray_backproject(w, rec)
        p_big, b_big = ctx.ray_project(d, rec, max_nodes=20000), ctx.ray_backproject(w, rec, max_nodes=20000)
        assert ctx.pool_bytes > pool
    assert _bits_equal(p_big.values, p_small.values) and (p_big.length == p_small.length).all()
    assert b_big.quantum_exp == b_small.quantum_exp and _bits_equal(b_big.grad, b_small.grad)


@gpu
def test_projection_over_a_source_range_is_a_slice_of_the_full_call():
    ms = _golden_cases()["hetero_818"]
    dims = tuple(ms[0]["dims"])
    rec = all_nodes(dims)[::7]
    d = np.random.default_rng(3).standard_normal(dims).astype(np.float32)
    ctx, v = _ctx(ms)
    with ctx:
        full = ctx.ray_project(d, rec)
        parts = [ctx.ray_project(d, rec, sources=range(s, s + 1)) for s in range(3)]
        tail = ctx.ray_project(d, rec, sources=(1, 2))
        with pytest.raises(P.SweepError, match="not within"):
            ctx.ray_project(d, rec, sources=(2, 2))
        with pytest.raises(P.SweepError, match="shape"):
            ctx.ray_project(d[:-1], rec)
    for s, part in enumerate(parts):
        assert _bits_equal(part.values[0], full.values[s]) and (part.status[0] == full.status[s]).all()
    assert _bits_equal(tail.values, full.values[1:]) and (tail.length == full.length[1:]).all()


@gpu
def test_full_size_config2_projection_and_coverage():
    v = W.heterogeneous_field((241, 241, 51), seed=7)
    star = W.star("818")
    gold = [g for g in json.loads((ROOT / "tests" / "golden" / "full_241.json").read_text())
            if g["label"].startswith("config2")]
    assert hashlib.sha256(v.tobytes()).hexdigest() == gold[0]["v_sha256"]
    starts = [g["start"] for g in gold]
    face = np.array([(x, y, 0) for x in range(241) for y in range(241)], np.int32)
    rng = np.random.default_rng(2025)
    pick = np.sort(rng.choice(len(face), 300, replace=False))
    with P.SweepContext(kernel=api.KERNEL_TILED) as ctx:
        ctx.set_model(v); ctx.set_star(star); ctx.set_sources(starts)
        ctx.run()
        fields = [ctx.get_tt(s) for s in range(len(starts))]
        proj = ctx.ray_project(v, face)
        cov = ctx.ray_backproject(np.ones((len(starts), len(pick)), np.float32), face[pick])
    rays = []
    for s, (g, tt) in enumerate(zip(gold, fields)):
        assert hashlib.sha256(tt.tobytes()).hexdigest() == g["tt_sha256"], f"{g['label']}: field differs"
        assert (proj.status[s] == OK).all()
        assert _bits_equal(proj.values[s], tt[:, :, 0].ravel()), g["label"]
        nodes, length, status, _ = oracle_rays(v, tt, star, g["start"], face[pick])
        rays.append((nodes, length, status))
    want, e = oracle_backproject(v.shape, rays, np.ones((len(starts), len(pick)), np.float32), _hd_max("818"))
    assert cov.quantum_exp == e and _bits_equal(cov.grad, want)


@gpu
def test_misfit_gradient():
    ms = _golden_cases()["hetero_818"]
    dims = tuple(ms[0]["dims"])
    v = make_field(ms[0]["kind"], dims, ms[0]["seed"])
    star = W.star("818")
    starts = [m["start"] for m in ms]
    rec = all_nodes(dims)[::11]
    t = np.stack([m["tt"].ravel()[np.ravel_multi_index(tuple(rec.T), dims)] for m in ms])
    same = P.misfit_gradient(v, star, starts, rec, t)
    assert same.misfit == 0.0 and same.quantum_exp == 0
    assert (same.gradient.view(np.uint32) == 0).all(), "observed = predicted: the gradient is all +0"
    rng = np.random.default_rng(6)
    obs = (t * rng.uniform(0.97, 1.03, t.shape)).astype(np.float32)
    obs[rng.random(obs.shape) < 0.1] = np.nan   # no pick
    mg = P.misfit_gradient(v, star, starts, rec, obs)
    use = ~np.isnan(obs)
    assert (mg.status == OK).all()
    want_res = np.where(use, (t - obs).astype(np.float32), np.float32(np.nan))
    assert _bits_equal(mg.residual, want_res)
    assert mg.misfit == 0.5 * float(np.sum(want_res[use].astype(np.float64) ** 2)) and mg.misfit > 0
    with P.SweepContext() as ctx:
        ctx.set_model(v); ctx.set_star(star); ctx.set_sources(starts); ctx.run()
        bp = ctx.ray_backproject(np.nan_to_num(mg.residual, nan=0.0), rec)
    assert bp.quantum_exp == mg.quantum_exp and _bits_equal(bp.grad, mg.gradient)
