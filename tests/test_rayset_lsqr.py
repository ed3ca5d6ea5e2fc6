"""The damped and smoothed LSQR step of a ray set, solved on the device (include/sweeptt.h, sweeptt_rayset_lsqr).

The yardstick is lsqr_restated: scipy's lsqr restated statement for statement in numpy / float64 scalars, with every
norm sqrt(sumsq(v)) in the documented fixed order and the first-difference rows D appended to G.  CPU: the restatement
agrees with scipy's lsqr on the explicit float64 [G; smooth D] within the Golub-Van Loan bound; D and D^T are adjoint;
sumsq equals its literal definition; the new kernels never fuse a multiply-add; a C99 client links.  GPU (-m gpu):
RaySet.lsqr equals the restatement bit for bit (x, istop, itn and the six norms) on the golden cases, with and without
damping and smoothing, on subsets of rows, truncated sets, every stopping reason and every axis permutation; full-size
config 2; determinism, the reduction grid, the set and the context left unchanged, memory released; every refusal;
and smoothing lowers the roughness of the update."""
import hashlib
import json
import math
import re
import shutil
import subprocess

import numpy as np
import pytest
import torch
from scipy.sparse.linalg import lsqr

import uoparallel_seismic_project_b200 as P
from uoparallel_seismic_project_b200 import api, workloads as W

from conftest import ROOT, make_field
from test_rays import _golden_cases, _oracle_rays, all_nodes
from test_rayset import _case_problem, explicit_g, oracle_operator
from test_tomography import _bits_equal, _ctx, _hd_max

gpu = pytest.mark.gpu
OK, TRUNCATED = api.RAY_OK, api.RAY_TRUNCATED
U = 2.0 ** -24   # unit roundoff of float32
BLOCK = 2048


# ---- the restatement ---------------------------------------------------------------------------

def sumsq(v):
    """Squares, padded with +0 to a multiple of 2048, every block summed by the halving tree a[i] + a[i+h],
    h = 1024 .. 1; the same tree over the block sums until one value is left.  sumsq of nothing is +0."""
    a = np.asarray(v, np.float64).ravel()
    a = a * a
    if a.size == 0:
        return np.float64(0.0)
    while True:
        nb = -(-a.size // BLOCK)
        a = np.concatenate([a, np.zeros(nb * BLOCK - a.size)]).reshape(nb, BLOCK)
        h = BLOCK // 2
        while h:
            a = a[:, :h] + a[:, h:2 * h]
            h //= 2
        a = a[:, 0]
        if a.size == 1:
            return a[0]


def sumsq_literal(v):
    """The definition word for word, on Python floats."""
    def tree(block):
        a = list(block) + [0.0] * (BLOCK - len(block))
        h = BLOCK // 2
        while h:
            for i in range(h):
                a[i] = a[i] + a[i + h]
            h //= 2
        return a[0]

    def level(xs):
        sums = [tree(xs[i:i + BLOCK]) for i in range(0, len(xs), BLOCK)]
        return sums[0] if len(sums) == 1 else level(sums)

    xs = [float(x) * float(x) for x in np.asarray(v, np.float64).ravel()]
    return level(xs) if xs else 0.0


def d_rows(x, dims, smooth):
    """D x: for axis 0, 1, 2 the rows fl(smooth * fl(x[n+e_a] - x[n])), n in FLOATBOX order."""
    x = np.asarray(x, np.float64).reshape(dims)
    return np.concatenate([smooth * np.diff(x, axis=a).ravel() for a in range(3)])


def d_count(dims):
    nx, ny, nz = dims
    return (nx - 1) * ny * nz + nx * (ny - 1) * nz + nx * ny * (nz - 1)


def dt_cols(y, dims, smooth):
    """D^T y: acc = +0; for a = 0, 1, 2: + y_a[j - e_a] where that node is in the box, then - y_a[j] where j + e_a is;
    fl(smooth * acc)."""
    acc = np.zeros(dims)
    off = 0
    for a in range(3):
        shape = list(dims)
        shape[a] -= 1
        cnt = int(np.prod(shape))
        ya = np.asarray(y[off:off + cnt], np.float64).reshape(shape)
        off += cnt
        hi = tuple(slice(1, None) if k == a else slice(None) for k in range(3))
        lo = tuple(slice(None, -1) if k == a else slice(None) for k in range(3))
        acc[hi] = acc[hi] + ya
        acc[lo] = acc[lo] - ya
    return (smooth * acc).ravel()


def sym_ortho(a, b):
    sign = np.sign
    if b == 0:
        return sign(a), np.float64(0), abs(a)
    if a == 0:
        return np.float64(0), sign(b), abs(b)
    if abs(b) > abs(a):
        tau = a / b
        s = sign(b) / np.sqrt(1 + tau * tau)
        c = s * tau
        return c, s, b / s
    tau = b / a
    c = sign(a) / np.sqrt(1 + tau * tau)
    s = c * tau
    return c, s, a / c


def lsqr_restated(matvec, rmatvec, b, dims, *, damp=0.0, smooth=0.0, atol=1e-6, btol=1e-6, conlim=1e8, iter_lim=None):
    """scipy 1.18's lsqr (x0 = None, calc_var = False) on A = [G; smooth D], statement for statement, with every square
    x*x and every norm sqrt(sumsq(.)).  matvec / rmatvec apply G and G^T in float64.  Returns scipy's tuple without
    var: (x, istop, itn, r1norm, r2norm, anorm, acond, arnorm, xnorm)."""
    f = np.float64
    n = int(np.prod(dims))
    b = np.asarray(b, np.float64).ravel()
    m = b.size
    iter_lim = 2 * n if iter_lim is None else iter_lim
    damp, atol, btol, conlim = f(damp), f(atol), f(btol), f(conlim)
    eps = f(np.finfo(np.float64).eps)

    def A(v):
        out = np.asarray(matvec(v), np.float64)
        return np.concatenate([out, d_rows(v, dims, smooth)]) if smooth > 0 else out

    def AT(u):
        g = np.asarray(rmatvec(u[:m]), np.float64)
        return g + dt_cols(u[m:], dims, smooth) if smooth > 0 else g

    def norm(v):
        return np.sqrt(sumsq(v))

    with np.errstate(all="ignore"):
        itn, istop = 0, 0
        ctol = f(0)
        if conlim > 0:
            ctol = 1 / conlim
        anorm = acond = ddnorm = res2 = xnorm = xxnorm = z = f(0)
        dampsq = damp * damp
        cs2, sn2 = f(-1), f(0)
        u = np.concatenate([b, np.zeros(d_count(dims) if smooth > 0 else 0)])
        bnorm = norm(u)
        x = np.zeros(n)
        beta = bnorm
        if beta > 0:
            u = (1 / beta) * u
            v = AT(u)
            alfa = norm(v)
        else:
            v = x.copy()
            alfa = f(0)
        if alfa > 0:
            v = (1 / alfa) * v
        w = v.copy()
        rhobar, phibar = alfa, beta
        rnorm = r1norm = r2norm = beta
        arnorm = alfa * beta
        if arnorm == 0:
            return x, istop, itn, r1norm, r2norm, anorm, acond, arnorm, xnorm
        while itn < iter_lim:
            itn = itn + 1
            u = A(v) - alfa * u
            beta = norm(u)
            if beta > 0:
                u = (1 / beta) * u
                anorm = np.sqrt(anorm * anorm + alfa * alfa + beta * beta + dampsq)
                v = AT(u) - beta * v
                alfa = norm(v)
                if alfa > 0:
                    v = (1 / alfa) * v
            if damp > 0:
                rhobar1 = np.sqrt(rhobar * rhobar + dampsq)
                cs1 = rhobar / rhobar1
                sn1 = damp / rhobar1
                psi = sn1 * phibar
                phibar = cs1 * phibar
            else:
                rhobar1 = rhobar
                psi = f(0)
            cs, sn, rho = sym_ortho(rhobar1, beta)
            theta = sn * alfa
            rhobar = -cs * alfa
            phi = cs * phibar
            phibar = sn * phibar
            tau = sn * phi
            t1 = phi / rho
            t2 = -theta / rho
            dk = (1 / rho) * w
            x = x + t1 * w
            w = v + t2 * w
            dkn = norm(dk)
            ddnorm = ddnorm + dkn * dkn
            delta = sn2 * rho
            gambar = -cs2 * rho
            rhs = phi - delta * z
            zbar = rhs / gambar
            xnorm = np.sqrt(xxnorm + zbar * zbar)
            gamma = np.sqrt(gambar * gambar + theta * theta)
            cs2 = gambar / gamma
            sn2 = theta / gamma
            z = rhs / gamma
            xxnorm = xxnorm + z * z
            acond = anorm * np.sqrt(ddnorm)
            res1 = phibar * phibar
            res2 = res2 + psi * psi
            rnorm = np.sqrt(res1 + res2)
            arnorm = alfa * abs(tau)
            if damp > 0:
                r1sq = rnorm * rnorm - dampsq * xxnorm
                r1norm = np.sqrt(abs(r1sq))
                if r1sq < 0:
                    r1norm = -r1norm
            else:
                r1norm = rnorm
            r2norm = rnorm
            test1 = rnorm / bnorm
            test2 = arnorm / (anorm * rnorm + eps)
            test3 = 1 / (acond + eps)
            t1 = test1 / (1 + anorm * xnorm / bnorm)
            rtol = btol + atol * anorm * xnorm / bnorm
            if itn >= iter_lim:
                istop = 7
            if 1 + test3 <= 1:
                istop = 6
            if 1 + test2 <= 1:
                istop = 5
            if 1 + t1 <= 1:
                istop = 4
            if test3 <= ctol:
                istop = 3
            if test2 <= atol:
                istop = 2
            if test1 <= rtol:
                istop = 1
            if istop != 0:
                break
    return x, istop, itn, r1norm, r2norm, anorm, acond, arnorm, xnorm


def set_operator(rs, rows):
    """G_rows from the set's own host calls, with as_linear_operator's conversions."""
    op = rs.as_linear_operator(rows)
    return op.matvec, op.rmatvec


def _golden_problem(case, missing=0.0, seed=6):
    """Rows (OK rays with a pick; `missing` of the picks removed), b = float64(float32(observed - t)) over them."""
    ms, rays, t, obs = _case_problem(case, seed)
    obs = obs.copy()
    obs[np.random.default_rng(seed + 1).random(obs.shape) < missing] = np.nan
    status = np.stack([r[2] for r in rays])
    residual = (obs - t).astype(np.float32)
    rows = np.isfinite(residual) & (status == OK)
    return ms, rays, rows, residual[rows].astype(np.float64)


def assert_same_solution(got, want, what):
    x, *scalars = want
    names = ["istop", "itn", "r1norm", "r2norm", "anorm", "acond", "arnorm", "xnorm"]
    for name, w in zip(names, scalars):
        g = getattr(got, name)
        assert (g == w) if name in ("istop", "itn") else np.float64(g).view(np.uint64) == np.float64(w).view(np.uint64), \
            f"{what}: {name} {g!r} != {w!r}"
    nd = int((got.x.ravel().view(np.uint64) != np.asarray(x, np.float64).view(np.uint64)).sum())
    assert nd == 0, f"{what}: x differs in {nd} nodes"


# ---- CPU ---------------------------------------------------------------------------------------

@pytest.mark.parametrize("smooth", [0.0, 3.0])
def test_restatement_agrees_with_scipy_on_the_explicit_matrix(smooth):
    """As test_lsqr_reference_agrees_with_lsqr_on_the_explicit_matrix, with the smoothing rows: both runs converge
    (atol = btol = 1e-10) on A = [G; smooth D; damp I]; the float32 operators perturb G by eps = (L_max + 2) u per entry
    (D is applied in float64), so |dx|/|x| <= eps kappa (2 + kappa |res| / (|A| |x|)) (Golub & Van Loan, Thm. 5.3.1)."""
    damp = 20.0
    ms, rays, rows, b = _golden_problem("rand_818")
    dims = tuple(ms[0]["dims"])
    op = oracle_operator(dims, rays, rows, _hd_max(ms[0]["star"]))
    out = lsqr_restated(op.matvec, op.rmatvec, b, dims, damp=damp, smooth=smooth, atol=1e-10, btol=1e-10, iter_lim=400)
    G = explicit_g(dims, rays, rows)
    n = G.shape[1]
    if smooth > 0:
        Dm = np.stack([d_rows(e, dims, 1.0) for e in np.eye(n)], axis=1)
        G = np.vstack([G, smooth * Dm])
    bb = np.concatenate([b, np.zeros(G.shape[0] - b.size)])
    ref = lsqr(G, bb, damp=damp, atol=1e-10, btol=1e-10, iter_lim=400)
    assert out[1] in (1, 2) and ref[1] in (1, 2), (out[1], ref[1])
    sv = np.linalg.svd(G, compute_uv=False)
    norm_a = np.hypot(sv[0], damp)
    kappa = norm_a / np.hypot(sv[-1], damp)
    A = np.vstack([G, damp * np.eye(n)])
    rhs = np.concatenate([bb, np.zeros(n)])
    x = np.linalg.lstsq(A, rhs, rcond=None)[0]
    res = np.linalg.norm(rhs - A @ x)
    eps = (max(int(r[1].max()) for r in rays) + 2) * U
    tol = eps * kappa * (2 + kappa * res / (norm_a * np.linalg.norm(x)))
    err = np.linalg.norm(out[0] - ref[0]) / np.linalg.norm(ref[0])
    assert err <= tol, (err, tol, kappa)


def test_restated_d_and_dt_are_adjoint():
    rng = np.random.default_rng(3)
    for dims in [(12, 11, 9), (1, 5, 7), (4, 1, 1), (1, 1, 1), (3, 2, 1)]:
        x = rng.standard_normal(dims)
        y = rng.standard_normal(d_count(dims))
        lhs, rhs = float(d_rows(x, dims, 1.5) @ y), float(x.ravel() @ dt_cols(y, dims, 1.5))
        scale = 1.5 * (np.abs(x).sum() * np.abs(y).max(initial=0) * 2 + 1)
        assert abs(lhs - rhs) <= 8 * x.size * 2.0 ** -53 * scale, (dims, lhs, rhs)
        assert d_rows(x, dims, 1.5).size == d_count(dims)


@pytest.mark.parametrize("length", [0, 1, 2047, 2048, 2049, BLOCK * BLOCK + 1])
def test_sumsq_follows_its_definition(length):
    rng = np.random.default_rng(length)
    v = rng.uniform(0.5, 1.0, length) * 2.0 ** rng.integers(-540, 250, length) * rng.choice([-1, 1], length)
    if length > 4:
        v[:4] = [5e-324, -2.0 ** -1074 * 3, 1e150, -0.0]
    got = sumsq(v)
    assert np.float64(got).view(np.uint64) == np.float64(sumsq_literal(v)).view(np.uint64)
    exact = math.fsum(float(x) * float(x) for x in v)   # the squares are rounded once; fsum sums them exactly
    sq = [float(x) * float(x) for x in v]
    bound = (math.log2(max(length, 1)) + 1) * 2.0 ** -53 * math.fsum(sq)
    assert abs(float(got) - exact) <= bound, (got, exact, bound)


@pytest.mark.skipif(shutil.which("cuobjdump") is None, reason="cuobjdump not on PATH")
def test_lsqr_kernels_never_fuse_multiply_add():
    out = subprocess.run(["cuobjdump", "-sass", str(P.lib_path())], capture_output=True, text=True, check=True).stdout
    funcs, name = {}, None
    for line in out.splitlines():
        mm = re.search(r"Function : (\S+)", line)
        if mm:
            name = mm.group(1)
            funcs[name] = []
        elif name and re.match(r"\s+/\*[0-9a-f]{4,6}\*/", line):
            funcs[name].append(line)
    kernels = {k: v for k, v in funcs.items() if "lsqr_" in k}
    assert len(kernels) == 8, sorted(kernels)
    for k, lines in kernels.items():
        text = "\n".join(lines)
        assert not re.search(r"\b[DF]FMA2?\b", text), f"{k}: fused multiply-add found"
    assert all("DADD" in "\n".join(v) for k, v in kernels.items() if re.search(r"lsqr_(u|v|xw|reduce|sumsq)_kernel", k))


def test_c99_client_links_against_rayset_lsqr(tmp_path):
    """Without a GPU the call fails with a message; with one, on a tiny constant box, the solve of G x = b for the one
    ray's time has x > 0 along the ray, and a refused call names its reason."""
    src = tmp_path / "client.c"
    src.write_text(r'''
#include <stdio.h>
#include "sweeptt.h"
int main(void) {
  struct FS fs[7] = {{1, 0, 0, 0.f}, {-1, 0, 0, 0.f}, {0, 1, 0, 0.f}, {0, -1, 0, 0.f}, {0, 0, 1, 0.f},
                     {0, 0, -1, 0.f}, {1, 1, 1, 0.f}};
  struct START st[1] = {{0, 0, 0}}, rec[1] = {{3, 0, 0}};
  float v[64];
  double b[1] = {30.0}, x[64];
  int i;
  sweeptt_lsqr_opts opts = {sizeof(sweeptt_lsqr_opts), 0.0, 0.5, 1e-6, 1e-6, 1e8, 50};
  sweeptt_lsqr_info info = {sizeof(sweeptt_lsqr_info), 0, 0, 0., 0., 0., 0., 0., 0.};
  sweeptt_stats stats;
  sweeptt_ctx *ctx;
  sweeptt_rayset *set;
  for (i = 0; i < 64; i++) v[i] = 1.f;
  sweeptt_star_fill_distances(fs, 7, 10.0f);
  ctx = sweeptt_create(NULL);
  if (!ctx) {
    if (sweeptt_rayset_lsqr(NULL, NULL, b, &opts, x, &info, &stats)) return 2;
    printf("%s\n", sweeptt_last_error());
    return 0;
  }
  if (!sweeptt_set_model(ctx, v, 4, 4, 4) || !sweeptt_set_star(ctx, fs, 7) || !sweeptt_set_sources(ctx, st, 1) ||
      !sweeptt_run(ctx, NULL) || !(set = sweeptt_rayset_freeze(ctx, 0, 1, rec, 1, 16, &stats)) ||
      !sweeptt_rayset_lsqr(set, NULL, b, &opts, x, &info, &stats)) {
    printf("%s\n", sweeptt_last_error());
    return 3;
  }
  if (info.itn < 1 || info.istop < 1 || !(x[0] > 0) || !(x[48] > 0) || stats.kernel_launches < 1) return 4;
  opts.damp = -1.0;
  if (sweeptt_rayset_lsqr(set, NULL, b, &opts, x, &info, &stats)) return 5;
  printf("%s\n", sweeptt_last_error());
  sweeptt_rayset_destroy(set);
  sweeptt_destroy(ctx);
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
        assert "ok" in r.stdout and "damp" in r.stdout, r.stdout
    else:
        assert "null ray set" in r.stdout, r.stdout


# ---- GPU ---------------------------------------------------------------------------------------

def _golden_set(case, **kw):
    ms = _golden_cases()[case]
    ctx, v = _ctx(ms, **kw)
    return ctx, ctx.freeze_rays(all_nodes(tuple(ms[0]["dims"])))


@gpu
@pytest.mark.parametrize("case", ["rand_818", "hetero_818"])
@pytest.mark.parametrize("damp", [0.0, 20.0])
@pytest.mark.parametrize("smooth", [0.0, 3.0])
def test_lsqr_equals_the_restatement_on_the_oracle_operators(case, damp, smooth):
    iters = 25 if case == "rand_818" else 10
    ms, rays, rows, b = _golden_problem(case, missing=0.1 if case == "hetero_818" else 0.0)
    dims = tuple(ms[0]["dims"])
    op = oracle_operator(dims, rays, rows, _hd_max(ms[0]["star"]))
    want = lsqr_restated(op.matvec, op.rmatvec, b, dims, damp=damp, smooth=smooth, iter_lim=iters)
    ctx, rs = _golden_set(case)
    with ctx, rs:
        assert (rs.status == np.stack([r[2] for r in rays])).all()
        got = rs.lsqr(b, rows, damp=damp, smooth=smooth, iter_lim=iters)
    assert_same_solution(got, want, f"{case} damp={damp} smooth={smooth}")
    assert got.stats.solve_ms > 0 and got.stats.kernel_launches > 10 * got.itn
    assert got.stats.h2d_bytes == 16 * b.size and got.stats.d2h_bytes >= 8 * int(np.prod(dims))


@gpu
@pytest.mark.parametrize("axis", ["0", "1", "2"])
def test_lsqr_does_not_depend_on_the_axis_permutation(axis, monkeypatch):
    monkeypatch.setenv("SWEEPTT_WINDOW_AXIS", axis)
    ms, rays, rows, b = _golden_problem("rand_818")
    dims = tuple(ms[0]["dims"])
    op = oracle_operator(dims, rays, rows, _hd_max(ms[0]["star"]))
    want = lsqr_restated(op.matvec, op.rmatvec, b, dims, damp=2.0, smooth=3.0, iter_lim=15)
    ctx, rs = _golden_set("rand_818")
    with ctx, rs:
        got = rs.lsqr(b, rows, damp=2.0, smooth=3.0, iter_lim=15)
    assert_same_solution(got, want, f"axis {axis}")


@gpu
def test_lsqr_stopping_reasons_and_truncated_sets():
    ms, rays, rows, b = _golden_problem("rand_818")
    dims = tuple(ms[0]["dims"])
    op = oracle_operator(dims, rays, rows, _hd_max(ms[0]["star"]))
    ctx, rs = _golden_set("rand_818")
    with ctx, rs:
        for kw, stops in [(dict(damp=20.0, atol=1e-3, btol=1e-3, iter_lim=300), (1, 2)),
                          (dict(damp=0.0, smooth=3.0, atol=1e-3, btol=1e-3, iter_lim=300), (1, 2)),
                          (dict(damp=1.0, iter_lim=4), (7,)),
                          (dict(damp=1.0, conlim=2.0, iter_lim=300), (3,))]:
            want = lsqr_restated(op.matvec, op.rmatvec, b, dims, **kw)
            assert want[1] in stops, (kw, want[1])
            assert_same_solution(rs.lsqr(b, rows, **kw), want, str(kw))
        zero = rs.lsqr(np.zeros_like(b), rows, damp=1.0, smooth=3.0)
        assert zero.istop == 0 and zero.itn == 0 and not zero.x.any() and zero.r1norm == 0
        assert_same_solution(zero, lsqr_restated(op.matvec, op.rmatvec, 0 * b, dims, damp=1.0, smooth=3.0), "b = 0")
        with ctx.freeze_rays(all_nodes(dims), max_nodes=3) as short:
            assert (short.status == TRUNCATED).any() and (short.status == OK).any()
            sel = short.status == OK
            bs = np.random.default_rng(4).standard_normal(int(sel.sum()))
            for smooth in (0.0, 3.0):
                want = lsqr_restated(*set_operator(short, sel), bs, dims, damp=1.0, smooth=smooth, iter_lim=12)
                assert_same_solution(short.lsqr(bs, damp=1.0, smooth=smooth, iter_lim=12), want, f"truncated {smooth}")


@gpu
def test_lsqr_is_deterministic_and_leaves_the_set_and_context_unchanged(monkeypatch):
    ms, rays, rows, b = _golden_problem("hetero_818", missing=0.1)
    dims = tuple(ms[0]["dims"])
    d = np.random.default_rng(11).standard_normal(dims).astype(np.float32)
    w = np.random.default_rng(12).standard_normal((len(ms), int(np.prod(dims)))).astype(np.float32)
    ctx, rs = _golden_set("hetero_818")
    with ctx, rs:
        fields = [ctx.get_tt(s) for s in range(len(ms))]
        p0, g0 = rs.project(d), rs.backproject(w)
        first = rs.lsqr(b, rows, damp=1.0, smooth=2.0, iter_lim=12)
        again = rs.lsqr(b, rows, damp=1.0, smooth=2.0, iter_lim=12)
        for ctas in ("1", "3", "100000"):
            monkeypatch.setenv("SWEEPTT_LSQR_CTAS", ctas)
            other = rs.lsqr(b, rows, damp=1.0, smooth=2.0, iter_lim=12)
            assert_same_solution(other, (first.x.ravel(), first.istop, first.itn, first.r1norm, first.r2norm,
                                         first.anorm, first.acond, first.arnorm, first.xnorm), f"ctas {ctas}")
        monkeypatch.delenv("SWEEPTT_LSQR_CTAS")
        assert_same_solution(again, (first.x.ravel(), first.istop, first.itn, first.r1norm, first.r2norm, first.anorm,
                                     first.acond, first.arnorm, first.xnorm), "second call")
        p1, g1 = rs.project(d), rs.backproject(w)
        assert _bits_equal(p0.values, p1.values) and _bits_equal(g0.grad, g1.grad) and g0.quantum_exp == g1.quantum_exp
        assert all(_bits_equal(f, ctx.get_tt(s)) for s, f in enumerate(fields))


@gpu
def test_lsqr_refusals_leave_the_set_working():
    ms, rays, rows, b = _golden_problem("rand_818")
    ctx, rs = _golden_set("rand_818")
    with ctx, rs:
        want = rs.lsqr(b, rows, damp=1.0, smooth=1.0, iter_lim=5)
        with ctx.freeze_rays(all_nodes(tuple(ms[0]["dims"])), max_nodes=3) as short:
            sel = short.status != OK
            with pytest.raises(P.SweepError, match="not OK"):
                short.lsqr(np.ones(int(sel.sum())), sel)
        nan_b = b.copy()
        nan_b[7] = np.nan
        with pytest.raises(P.SweepError, match=r"b\[7\] is not finite"):
            rs.lsqr(nan_b, rows)
        inf_b = b.copy()
        inf_b[0] = -np.inf
        with pytest.raises(P.SweepError, match="not finite"):
            rs.lsqr(inf_b, rows)
        for kw, msg in [(dict(damp=-1.0), "damp"), (dict(damp=np.inf), "damp"), (dict(damp=np.nan), "damp"),
                        (dict(smooth=-0.5), "smooth"), (dict(smooth=np.inf), "smooth"),
                        (dict(atol=-1e-6), "atol"), (dict(btol=-1.0), "btol"), (dict(conlim=-1.0), "conlim"),
                        (dict(atol=np.nan), "atol"), (dict(iter_lim=-1), "iter_lim")]:
            with pytest.raises(P.SweepError, match=msg):
                rs.lsqr(b, rows, **kw)
        lib = api.load_library()
        x = np.empty(rs.dims, np.float64)
        sel = np.ascontiguousarray(rows, np.uint8)
        good = api._LsqrOpts(api.C.sizeof(api._LsqrOpts), 1.0, 1.0, 1e-6, 1e-6, 1e8, 5)
        for opts, info in [(api._LsqrOpts(8, 1.0, 1.0, 1e-6, 1e-6, 1e8, 5), None),
                           (good, api._LsqrInfo(4))]:
            assert not lib.sweeptt_rayset_lsqr(rs._h, sel.ctypes.data, b.ctypes.data, api.C.byref(opts),
                                               x.ctypes.data, api.C.byref(info) if info else None, None)
            assert "struct_size" in lib.sweeptt_last_error().decode()
        for args in [(sel.ctypes.data, None, api.C.byref(good), x.ctypes.data),
                     (sel.ctypes.data, b.ctypes.data, None, x.ctypes.data),
                     (sel.ctypes.data, b.ctypes.data, api.C.byref(good), None)]:
            assert not lib.sweeptt_rayset_lsqr(rs._h, *args, None, None)
            assert "required" in lib.sweeptt_last_error().decode()
        assert not lib.sweeptt_rayset_lsqr(None, None, b.ctypes.data, api.C.byref(good), x.ctypes.data, None, None)
        assert "null ray set" in lib.sweeptt_last_error().decode()
        with pytest.raises(P.SweepError, match="b has"):
            rs.lsqr(b[:-1], rows)
        after = rs.lsqr(b, rows, damp=1.0, smooth=1.0, iter_lim=5)
        assert_same_solution(after, (want.x.ravel(), want.istop, want.itn, want.r1norm, want.r2norm, want.anorm,
                                     want.acond, want.arnorm, want.xnorm), "after the refusals")
    with pytest.raises(P.SweepError, match="closed"):
        rs.lsqr(b, rows)


@gpu
def test_smoothing_lowers_the_roughness_and_the_misfit():
    ms, rays, rows, b = _golden_problem("hetero_818", missing=0.1, seed=7)
    dims = tuple(ms[0]["dims"])
    ctx, rs = _golden_set("hetero_818")
    with ctx, rs:
        plain = rs.lsqr(b, rows, damp=1.0, iter_lim=30)
        smooth = rs.lsqr(b, rows, damp=1.0, smooth=5.0, iter_lim=30)
        for sol in (plain, smooth):
            gd = rs.project(sol.x.astype(np.float32)).values[rows].astype(np.float64)
            assert np.linalg.norm(b - gd) < np.linalg.norm(b), "the update lowers the linearised misfit"
    rough = [np.linalg.norm(d_rows(s.x, dims, 1.0)) for s in (plain, smooth)]
    assert rough[1] < rough[0], rough


@gpu
@pytest.mark.parametrize("smooth", [0.0, 1.0])
def test_full_size_config2_lsqr_equals_the_restatement(smooth):
    v = W.heterogeneous_field((241, 241, 51), seed=7)
    gold = [g for g in json.loads((ROOT / "tests" / "golden" / "full_241.json").read_text())
            if g["label"].startswith("config2")]
    assert hashlib.sha256(v.tobytes()).hexdigest() == gold[0]["v_sha256"]
    starts = [g["start"] for g in gold]
    face = np.array([(x, y, 0) for x in range(241) for y in range(241)], np.int32)
    with P.SweepContext(kernel=api.KERNEL_TILED) as ctx:
        ctx.set_model(v); ctx.set_star(W.star("818")); ctx.set_sources(starts)
        ctx.run()
        with ctx.freeze_rays(face) as rs:
            rows = rs.status == OK
            b = (rs.tt * np.random.default_rng(5).uniform(-0.02, 0.02, rs.shape)).astype(np.float32)[rows]
            b = b.astype(np.float64)
            rs.lsqr(b, damp=1.0, smooth=smooth, iter_lim=1)   # every kernel loaded before the memory is read
            torch.cuda.synchronize()
            free0 = torch.cuda.mem_get_info()[0]
            got = rs.lsqr(b, damp=1.0, smooth=smooth, atol=0.0, btol=0.0, iter_lim=20)
            free1 = torch.cuda.mem_get_info()[0]
            want = lsqr_restated(*set_operator(rs, rows), b, v.shape, damp=1.0, smooth=smooth, atol=0.0, btol=0.0,
                                 iter_lim=20)
            assert_same_solution(got, want, f"config 2, smooth {smooth}")
            assert got.itn == 20 and got.istop == 7
            if smooth == 0:
                ref = lsqr(rs.as_linear_operator(rows), b, damp=1.0, atol=0.0, btol=0.0, iter_lim=20)
                assert (ref[1], ref[2]) == (got.istop, got.itn)
                assert np.linalg.norm(ref[0] - got.x.ravel()) <= 1e-6 * np.linalg.norm(ref[0])
    assert free1 == free0, (free0, free1)
