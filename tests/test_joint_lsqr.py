"""Slowness and hypocentres solved together: the ray set's LSQR step with 4 columns per receiver
(include/sweeptt.h, sweeptt_rayset_lsqr_hypo), hypocentre_partials and joint_update.

The yardstick is lsqr_joint_restated: lsqr_restated (test_rayset_lsqr.py) over x = [model; hypo], with the header's
order of the hypocentre terms in A v and A^T u and every norm over the concatenation.  CPU: it agrees with scipy's lsqr
on the explicit float64 [G H; smooth D 0]; with h = 0 it is lsqr_restated bit for bit; the extra columns never raise
the converged r2norm; the partials rule on hand-made fields; the SASS of the touched and new kernels; a C99 client;
and a displaced-event case on the CPU oracles that fixes the recovery thresholds.  GPU (-m gpu): RaySet.lsqr(hypo=)
equals the restatement bit for bit (x, hypo, istop, itn and the six norms) on the golden cases, subsets, truncated
sets, reduction boundaries, reduction grids and axis permutations; h = 0 equals the plain call; refusals; memory;
hypocentre_partials against the rule on the context's fields; joint_update against its composition; full-size
config 2; and the displaced-event case on the device."""
import hashlib
import json
import re
import shutil
import subprocess
from types import SimpleNamespace

import numpy as np
import pytest
import torch
from scipy.sparse.linalg import lsqr

import oracle
import uoparallel_seismic_project_b200 as P
from uoparallel_seismic_project_b200 import api, workloads as W

from conftest import ROOT
from test_rays import _golden_cases, all_nodes, oracle_rays
from test_rayset import explicit_g, oracle_operator
from test_rayset_lsqr import (U, _golden_problem, _golden_set, assert_same_solution, d_count, d_rows, dt_cols,
                              lsqr_restated, set_operator, sumsq, sym_ortho)
from test_tomography import _hd_max

gpu = pytest.mark.gpu
OK, TRUNCATED = api.RAY_OK, api.RAY_TRUNCATED


# ---- the restatement ---------------------------------------------------------------------------

def hypo_terms(h, recv, nrec):
    """(A_H y, H^T u) of the hypocentre columns: row i (receiver recv[i]) adds fl(h[i, c] * y[recv[i], c]) to its G
    value for c = 0..3 in turn; column (r, c) of H^T u is acc = +0, acc = fl(acc + fl(h[i, c] u_i)) over the rows of r
    in increasing i."""
    h = np.asarray(h, np.float64).reshape(-1, 4)
    recv = np.asarray(recv, np.int64)
    order = np.argsort(recv, kind="stable")
    rank = np.empty(len(recv), np.int64)        # position of every row among the rows of its receiver
    if len(recv):
        starts = np.searchsorted(recv[order], recv[order])
        rank[order] = np.arange(len(recv)) - starts

    def av(g, y):
        y = y.reshape(nrec, 4)
        for c in range(4):
            g = g + h[:, c] * y[recv, c]
        return g

    def htu(u):
        acc = np.zeros((nrec, 4))
        for k in range(int(rank.max(initial=-1)) + 1):
            sel = rank == k
            acc[recv[sel]] = acc[recv[sel]] + h[sel] * u[sel][:, None]
        return acc.ravel()

    return av, htu


def lsqr_joint_restated(matvec, rmatvec, b, h, recv, nrec, dims, *, damp=0.0, smooth=0.0, atol=1e-6, btol=1e-6,
                        conlim=1e8, iter_lim=None):
    """lsqr_restated on A = [G H; smooth D 0] over x = [model (D values); hypo (4 nrec values)], statement for
    statement.  recv[i] is the receiver of row i.  Returns (x_model, istop, itn, r1norm, r2norm, anorm, acond, arnorm,
    xnorm, hypo [nrec, 4])."""
    f = np.float64
    n = int(np.prod(dims))
    nh = 4 * nrec
    b = np.asarray(b, np.float64).ravel()
    m = b.size
    iter_lim = 2 * n if iter_lim is None else iter_lim
    damp, atol, btol, conlim = f(damp), f(atol), f(btol), f(conlim)
    eps = f(np.finfo(np.float64).eps)
    h_av, h_tu = hypo_terms(h, recv, nrec)

    def A(v):
        out = h_av(np.asarray(matvec(v[:n]), np.float64), v[n:])
        return np.concatenate([out, d_rows(v[:n], dims, smooth)]) if smooth > 0 else out

    def AT(u):
        g = np.asarray(rmatvec(u[:m]), np.float64)
        if smooth > 0:
            g = g + dt_cols(u[m:], dims, smooth)
        return np.concatenate([g, h_tu(u[:m])])

    def norm(v):
        return np.sqrt(sumsq(v))

    def done(x):
        return x[:n], istop, itn, r1norm, r2norm, anorm, acond, arnorm, xnorm, x[n:].reshape(nrec, 4)

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
        x = np.zeros(n + nh)
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
            return done(x)
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
    return done(x)


def assert_same_joint(got, want, what):
    assert_same_solution(got, want[:9], what)
    assert got.hypo is not None and got.hypo.shape == want[9].shape, what
    nd = int((got.hypo.view(np.uint64) != np.asarray(want[9], np.float64).view(np.uint64)).sum())
    assert nd == 0, f"{what}: hypo differs in {nd} values"


def receivers_of(rows):
    """Receiver of every selected row of rows [S, R], in q order."""
    return np.nonzero(rows)[1]


def random_h(m, seed):
    """Finite h with zeros, both signs, and magnitudes from 1e-30 to 1e30."""
    rng = np.random.default_rng(seed)
    h = rng.standard_normal((m, 4)) * rng.choice([1.0, 1.0, 1.0, 1.0, 0.0, 1e-30, 1e30, -1e-30], (m, 4))
    h[rng.random((m, 4)) < 0.1] = 0.0
    if m:
        h[0] = [0.0, -0.0, 1e30, -1e-30]
    return h


def partials_rule(fields, centres):
    """float64[E, S, 3] from fields [S, nx, ny, nz] (float32): per axis fl(0.5 fl(t+ - t-)) with both neighbours in the
    box and finite, the one-sided difference with one, 0 with none; NaN everywhere when t0 = +inf."""
    fields = np.asarray(fields, np.float32)
    dims = fields.shape[1:]
    out = np.zeros((len(centres), len(fields), 3))
    for e, c in enumerate(np.asarray(centres)):
        for s, f in enumerate(fields):
            t0 = np.float64(f[tuple(c)])
            if np.isinf(t0):
                out[e, s] = np.nan
                continue
            for a in range(3):
                nb = {}
                for d in (-1, 1):
                    n = np.array(c)
                    n[a] += d
                    if 0 <= n[a] < dims[a] and np.isfinite(f[tuple(n)]):
                        nb[d] = np.float64(f[tuple(n)])
                if len(nb) == 2:
                    out[e, s, a] = 0.5 * (nb[1] - nb[-1])
                elif 1 in nb:
                    out[e, s, a] = nb[1] - t0
                elif -1 in nb:
                    out[e, s, a] = t0 - nb[-1]
    return out


class _FieldContext:
    """What hypocentre_partials reads from a SweepContext, over numpy fields: dims, and trace_rays(max_nodes=1).tt."""

    def __init__(self, fields):
        self.fields = np.asarray(fields, np.float32)
        self.dims = self.fields.shape[1:]

    def trace_rays(self, receivers, sources=None, max_nodes=None):
        assert sources is None and max_nodes == 1
        r = np.asarray(receivers)
        return SimpleNamespace(tt=self.fields[:, r[:, 0], r[:, 1], r[:, 2]])


def _bits(a):
    return np.ascontiguousarray(a, np.float64).view(np.uint64)


# ---- the displaced-event case ------------------------------------------------------------------
# A constant box (0.25, 818-FS), 14 stations at the corners and face centres, 6 events whose true node is the centre
# (12, 12, 12) and whose located node is one node off along +-each axis (every station >= 12 nodes away).  The picks
# are the true times with origin 0, the step starts from origin 0, damp = 1, up to 60 iterations.  On the CPU oracles
# the step converges (istop 2, 7 iterations) and moves every event back along its displaced axis, with the true sign,
# by 0.237 nodes (0.24 at damp 0.1 and 0.3 as well: the minimum-norm step puts most of the time change into the
# slowness columns), by at most 0.005 nodes along the other axes, and shifts the origin by 0.01.  The thresholds keep a
# margin around those values.
DISP_DIMS = (25, 25, 25)
DISP_TRUE = (12, 12, 12)
DISP_STATIONS = [(x, y, z) for x in (0, 24) for y in (0, 24) for z in (0, 24)] + \
    [(0, 12, 12), (24, 12, 12), (12, 0, 12), (12, 24, 12), (12, 12, 0), (12, 12, 24)]
DISP_DAMP, DISP_ITERS = 1.0, 60
DISP_ALONG = (0.2, 0.3)     # |shift| along the displaced axis
DISP_ACROSS = 0.01          # |shift| along the other axes


def _disp_events():
    cs, true = [], []
    for a in range(3):
        for d in (-1, 1):
            c = list(DISP_TRUE)
            c[a] += d
            cs.append(c)
            true.append(-d * np.eye(3)[a])
    return np.array(cs, np.int32), np.array(true)


def _check_disp(shift, true):
    for e, (s, t) in enumerate(zip(shift, true)):
        a = int(np.argmax(np.abs(t)))
        assert np.sign(s[a]) == np.sign(t[a]), (e, s, t)
        assert DISP_ALONG[0] <= abs(s[a]) <= DISP_ALONG[1], (e, s, t)
        assert all(abs(s[k]) <= DISP_ACROSS for k in range(3) if k != a), (e, s, t)


# ---- CPU ---------------------------------------------------------------------------------------

@pytest.mark.parametrize("smooth", [0.0, 3.0])
def test_joint_restatement_agrees_with_scipy_on_the_explicit_matrix(smooth):
    """As test_restatement_agrees_with_scipy_on_the_explicit_matrix, on [G H; smooth D 0]: H is applied in float64, so
    only G carries the float32 perturbation eps = (L_max + 2) u per entry, and the same Golub-Van Loan bound holds."""
    damp = 20.0
    ms, rays, rows, b = _golden_problem("rand_818")
    dims = tuple(ms[0]["dims"])
    nrec = rows.shape[1]
    recv = receivers_of(rows)
    h = np.random.default_rng(3).standard_normal((b.size, 4)) * 5.0
    op = oracle_operator(dims, rays, rows, _hd_max(ms[0]["star"]))
    out = lsqr_joint_restated(op.matvec, op.rmatvec, b, h, recv, nrec, dims, damp=damp, smooth=smooth, atol=1e-10,
                              btol=1e-10, iter_lim=600)
    G = explicit_g(dims, rays, rows)
    n = G.shape[1]
    H = np.zeros((b.size, 4 * nrec))
    for c in range(4):
        H[np.arange(b.size), 4 * recv + c] = h[:, c]
    A = np.hstack([G, H])
    if smooth > 0:
        Dm = np.stack([d_rows(e, dims, 1.0) for e in np.eye(n)], axis=1)
        A = np.vstack([A, np.hstack([smooth * Dm, np.zeros((Dm.shape[0], 4 * nrec))])])
    bb = np.concatenate([b, np.zeros(A.shape[0] - b.size)])
    ref = lsqr(A, bb, damp=damp, atol=1e-10, btol=1e-10, iter_lim=600)
    assert out[1] in (1, 2) and ref[1] in (1, 2), (out[1], ref[1])
    sv = np.linalg.svd(A, compute_uv=False)
    norm_a = np.hypot(sv[0], damp)
    kappa = norm_a / np.hypot(sv[-1] if A.shape[0] >= A.shape[1] else 0.0, damp)
    Ad = np.vstack([A, damp * np.eye(A.shape[1])])
    rhs = np.concatenate([bb, np.zeros(A.shape[1])])
    x = np.linalg.lstsq(Ad, rhs, rcond=None)[0]
    res = np.linalg.norm(rhs - Ad @ x)
    eps = (max(int(r[1].max()) for r in rays) + 2) * U
    tol = eps * kappa * (2 + kappa * res / (norm_a * np.linalg.norm(x)))
    got = np.concatenate([out[0], out[9].ravel()])
    err = np.linalg.norm(got - ref[0]) / np.linalg.norm(ref[0])
    assert err <= tol, (err, tol, kappa)


@pytest.mark.parametrize("smooth", [0.0, 3.0])
@pytest.mark.parametrize("damp", [0.0, 20.0])
def test_zero_h_is_the_plain_restatement_bit_for_bit(damp, smooth):
    ms, rays, rows, b = _golden_problem("rand_818", missing=0.1)
    dims = tuple(ms[0]["dims"])
    op = oracle_operator(dims, rays, rows, _hd_max(ms[0]["star"]))
    want = lsqr_restated(op.matvec, op.rmatvec, b, dims, damp=damp, smooth=smooth, iter_lim=8)
    got = lsqr_joint_restated(op.matvec, op.rmatvec, b, np.zeros((b.size, 4)), receivers_of(rows), rows.shape[1],
                              dims, damp=damp, smooth=smooth, iter_lim=8)
    assert (_bits(got[0]) == _bits(want[0])).all()
    assert got[1:3] == want[1:3]
    assert all(_bits(g) == _bits(w) for g, w in zip(got[3:9], want[3:9]))
    assert (_bits(got[9]) == 0).all(), "hypo is +0"


@pytest.mark.parametrize("smooth", [0.0, 3.0])
def test_the_extra_columns_never_raise_the_converged_residual(smooth):
    """The damped minimum over [x; y] is at most the one over x alone (y = 0 is feasible)."""
    ms, rays, rows, b = _golden_problem("rand_818")
    dims = tuple(ms[0]["dims"])
    op = oracle_operator(dims, rays, rows, _hd_max(ms[0]["star"]))
    kw = dict(damp=5.0, smooth=smooth, atol=1e-9, btol=1e-9, iter_lim=3000)
    plain = lsqr_restated(op.matvec, op.rmatvec, b, dims, **kw)
    h = np.random.default_rng(9).standard_normal((b.size, 4))
    joint = lsqr_joint_restated(op.matvec, op.rmatvec, b, h, receivers_of(rows), rows.shape[1], dims, **kw)
    assert plain[1] in (1, 2) and joint[1] in (1, 2), (plain[1], joint[1])
    assert joint[4] <= plain[4], (joint[4], plain[4])


def test_hypocentre_partials_follow_the_rule_on_hand_made_fields():
    """Interior, every box face, a one-node axis, +inf neighbours on one side and on both, and a +inf centre; both
    against numbers written out by hand and against partials_rule."""
    f = np.zeros((2, 5, 4, 1), np.float32)
    f[0] = (np.arange(5)[:, None, None] * 3.0 + np.arange(4)[None, :, None] * 0.5 ** 3).astype(np.float32)
    f[1] = f[0] ** 2 / 7
    f[1, 2, 2, 0] = np.inf          # centre (2, 2, 0) of station 1 unreached
    f[0, 3, 1, 0] = np.inf          # +inf on the +x side of (2, 1, 0)
    f[0, 1, 1, 0] = np.inf          # ... and on the -x side of (2, 1, 0) too
    f[0, 4, 2, 0] = np.inf          # +inf on the +x side of (3, 2, 0)
    centres = np.array([(2, 2, 0), (0, 0, 0), (4, 3, 0), (2, 1, 0), (3, 2, 0), (0, 2, 0), (2, 0, 0)])
    got = api.hypocentre_partials(_FieldContext(f), centres)
    assert got.shape == (7, 2, 3) and got.dtype == np.float64
    assert np.array_equal(got, partials_rule(f, centres), equal_nan=True)
    t = f[0].astype(np.float64)
    assert list(got[0, 0]) == [0.5 * (t[3, 2, 0] - t[1, 2, 0]), 0.5 * (t[2, 3, 0] - t[2, 1, 0]), 0.0]   # interior
    assert np.isnan(got[0, 1]).all()                                                                 # t0 = +inf
    assert list(got[1, 0]) == [t[1, 0, 0] - t[0, 0, 0], t[0, 1, 0] - t[0, 0, 0], 0.0]                # low faces
    assert list(got[2, 0]) == [t[4, 3, 0] - t[3, 3, 0], 0.0, 0.0]    # high faces; -y is +inf and +y outside
    assert got[3, 0, 0] == 0.0                                                                       # both +inf
    assert got[4, 0, 0] == t[3, 2, 0] - t[2, 2, 0]                                                   # +x is +inf
    assert got[5, 0, 0] == t[1, 2, 0] - t[0, 2, 0] and got[6, 0, 1] == t[2, 1, 0] - t[2, 0, 0]
    assert (got[~np.isnan(got[:, :, 2]), 2] == 0).all(), "a one-node axis has no derivative"
    with pytest.raises(P.SweepError, match="outside"):
        api.hypocentre_partials(_FieldContext(f), [(5, 0, 0)])


def test_displaced_events_are_moved_back_on_the_cpu_oracles():
    v = W.constant_field(DISP_DIMS, 0.25)
    star = W.star("818")
    fields = np.stack([oracle.solve(v, star, s)[0] for s in DISP_STATIONS])
    centres, true = _disp_events()
    rays = [oracle_rays(v, f, star, s, centres)[:3] for f, s in zip(fields, DISP_STATIONS)]
    status = np.stack([r[2] for r in rays])
    assert (status == OK).all()
    obs = fields[:, DISP_TRUE[0], DISP_TRUE[1], DISP_TRUE[2]][:, None].astype(np.float64)
    t = np.stack([f[tuple(centres.T)] for f in fields]).astype(np.float64)
    rows = status == OK
    b = (obs - 0.0 - t)[rows]
    d = partials_rule(fields, centres).transpose(1, 0, 2)[rows]
    h = np.concatenate([d, np.ones((len(d), 1))], axis=1)
    op = oracle_operator(DISP_DIMS, rays, rows, _hd_max(star))
    out = lsqr_joint_restated(op.matvec, op.rmatvec, b, h, receivers_of(rows), len(centres), DISP_DIMS,
                              damp=DISP_DAMP, iter_lim=DISP_ITERS)
    _check_disp(out[9][:, :3], true)


@pytest.mark.skipif(shutil.which("cuobjdump") is None, reason="cuobjdump not on PATH")
def test_hypo_and_touched_kernels_never_fuse_multiply_add():
    out = subprocess.run(["cuobjdump", "-sass", str(P.lib_path())], capture_output=True, text=True, check=True).stdout
    funcs, name = {}, None
    for line in out.splitlines():
        mm = re.search(r"Function : (\S+)", line)
        if mm:
            name = mm.group(1)
            funcs[name] = []
        elif name and re.match(r"\s+/\*[0-9a-f]{4,6}\*/", line):
            funcs[name].append(line)
    lsqr_names = sorted(re.search(r"lsqr_\w+_kernel", k).group(0) for k in funcs if "lsqr_" in k)
    assert lsqr_names == sorted(f"lsqr_{p}_kernel" for p in
                                ("reduce", "sumsq", "to_f32", "u", "scale_u", "v", "scale", "xw")), lsqr_names
    hypo = [k for k in funcs if re.search(r"hypo_[uv]_kernel", k)]
    assert len(hypo) == 2, hypo
    for k in hypo + [k for k in funcs if re.search(r"lsqr_(u|v|xw|scale)_kernel", k)]:
        text = "\n".join(funcs[k])
        assert not re.search(r"\b[DF]FMA2?\b", text), f"{k}: fused multiply-add found"
        assert "DMUL" in text, k


def test_c99_client_links_against_rayset_lsqr_hypo(tmp_path):
    """Without a GPU the call fails with a message; with one, on a tiny constant box, one ray's residual is split
    between the model and its receiver's origin-time column, and a NULL hypo_out is refused."""
    src = tmp_path / "client.c"
    src.write_text(r'''
#include <stdio.h>
#include "sweeptt.h"
int main(void) {
  struct FS fs[7] = {{1, 0, 0, 0.f}, {-1, 0, 0, 0.f}, {0, 1, 0, 0.f}, {0, -1, 0, 0.f}, {0, 0, 1, 0.f},
                     {0, 0, -1, 0.f}, {1, 1, 1, 0.f}};
  struct START st[1] = {{0, 0, 0}}, rec[1] = {{3, 0, 0}};
  float v[64];
  double b[1] = {30.0}, h[4] = {0.0, 0.0, 0.0, 1.0}, x[64], y[4];
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
    if (sweeptt_rayset_lsqr_hypo(NULL, NULL, b, h, &opts, x, y, &info, &stats)) return 2;
    printf("%s\n", sweeptt_last_error());
    return 0;
  }
  if (!sweeptt_set_model(ctx, v, 4, 4, 4) || !sweeptt_set_star(ctx, fs, 7) || !sweeptt_set_sources(ctx, st, 1) ||
      !sweeptt_run(ctx, NULL) || !(set = sweeptt_rayset_freeze(ctx, 0, 1, rec, 1, 16, &stats)) ||
      !sweeptt_rayset_lsqr_hypo(set, NULL, b, h, &opts, x, y, &info, &stats)) {
    printf("%s\n", sweeptt_last_error());
    return 3;
  }
  if (info.itn < 1 || info.istop < 1 || !(x[0] > 0) || !(y[3] > 0) || y[0] != 0.0 || stats.kernel_launches < 1)
    return 4;
  if (sweeptt_rayset_lsqr_hypo(set, NULL, b, h, &opts, x, NULL, &info, &stats)) return 5;
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
        assert "ok" in r.stdout and "hypo_out are required" in r.stdout, r.stdout
    else:
        assert "null ray set" in r.stdout, r.stdout


# ---- GPU ---------------------------------------------------------------------------------------

@gpu
@pytest.mark.parametrize("case", ["rand_818", "hetero_818"])
@pytest.mark.parametrize("damp", [0.0, 20.0])
@pytest.mark.parametrize("smooth", [0.0, 3.0])
def test_joint_lsqr_equals_the_restatement(case, damp, smooth):
    iters = 25 if case == "rand_818" else 10
    ms, rays, rows, b = _golden_problem(case, missing=0.1 if case == "hetero_818" else 0.0)
    dims = tuple(ms[0]["dims"])
    h = random_h(b.size, 21)
    op = oracle_operator(dims, rays, rows, _hd_max(ms[0]["star"]))
    want = lsqr_joint_restated(op.matvec, op.rmatvec, b, h, receivers_of(rows), rows.shape[1], dims, damp=damp,
                               smooth=smooth, iter_lim=iters)
    ctx, rs = _golden_set(case)
    with ctx, rs:
        got = rs.lsqr(b, rows, hypo=h, damp=damp, smooth=smooth, iter_lim=iters)
    assert_same_joint(got, want, f"{case} damp={damp} smooth={smooth}")
    m, R = b.size, rows.shape[1]
    assert got.stats.h2d_bytes == 16 * m + 40 * m + 8 * (R + 1)
    assert got.stats.d2h_bytes >= 8 * (int(np.prod(dims)) + 4 * R)


@gpu
def test_zero_h_equals_the_plain_call_and_truncated_sets():
    ms, rays, rows, b = _golden_problem("hetero_818", missing=0.1)
    ctx, rs = _golden_set("hetero_818")
    with ctx, rs:
        for kw in (dict(damp=0.0, iter_lim=12), dict(damp=1.0, smooth=2.0, iter_lim=12),
                   dict(damp=20.0, smooth=3.0, iter_lim=300)):
            plain = rs.lsqr(b, rows, **kw)
            zero = rs.lsqr(b, rows, hypo=np.zeros((b.size, 4)), **kw)
            assert_same_solution(zero, (plain.x.ravel(), plain.istop, plain.itn, plain.r1norm, plain.r2norm,
                                        plain.anorm, plain.acond, plain.arnorm, plain.xnorm), f"h = 0 {kw}")
            assert (_bits(zero.hypo) == 0).all() and plain.hypo is None
        dims = rs.dims
        with ctx.freeze_rays(all_nodes(dims), max_nodes=3) as short:
            assert (short.status == TRUNCATED).any() and (short.status == OK).any()
            sel = short.status == OK
            bs = np.random.default_rng(4).standard_normal(int(sel.sum()))
            h = random_h(bs.size, 5)
            for smooth in (0.0, 3.0):
                want = lsqr_joint_restated(*set_operator(short, sel), bs, h, receivers_of(sel), sel.shape[1], dims,
                                           damp=1.0, smooth=smooth, iter_lim=12)
                assert_same_joint(short.lsqr(bs, hypo=h, damp=1.0, smooth=smooth, iter_lim=12), want,
                                  f"truncated {smooth}")


@gpu
@pytest.mark.parametrize("axis", ["0", "1", "2"])
def test_joint_lsqr_does_not_depend_on_the_grid_or_the_axis_permutation(axis, monkeypatch):
    monkeypatch.setenv("SWEEPTT_WINDOW_AXIS", axis)
    ms, rays, rows, b = _golden_problem("rand_818")
    dims = tuple(ms[0]["dims"])
    h = random_h(b.size, 7)
    op = oracle_operator(dims, rays, rows, _hd_max(ms[0]["star"]))
    want = lsqr_joint_restated(op.matvec, op.rmatvec, b, h, receivers_of(rows), rows.shape[1], dims, damp=2.0,
                               smooth=3.0, iter_lim=15)
    ctx, rs = _golden_set("rand_818")
    with ctx, rs:
        for ctas in (None, "1", "2", "100000"):
            if ctas:
                monkeypatch.setenv("SWEEPTT_LSQR_CTAS", ctas)
            assert_same_joint(rs.lsqr(b, rows, hypo=h, damp=2.0, smooth=3.0, iter_lim=15), want,
                              f"axis {axis} ctas {ctas}")


@gpu
@pytest.mark.parametrize("dims,total", [((9, 9, 7), 2047), ((8, 8, 8), 2048), ((7, 7, 9), 2049),
                                        ((9, 9, 7), 2047 + 2048), ((8, 8, 8), 2048 + 2048)])
def test_joint_lsqr_at_the_reduction_boundaries(dims, total):
    """D + 4R = total: receivers with no row, one row and every row selected."""
    D = int(np.prod(dims))
    R = (total - D) // 4
    assert D + 4 * R == total
    v = W.random_field(dims, 3)
    nodes = all_nodes(dims)
    rec = nodes[np.random.default_rng(1).integers(0, D, R)] if R > D else nodes[:R]
    with P.SweepContext() as ctx:
        ctx.set_model(v); ctx.set_star(W.star("818")); ctx.set_sources([(0, 0, 0), tuple(d - 1 for d in dims),
                                                                        (dims[0] // 2, 0, dims[2] - 1)])
        ctx.run()
        with ctx.freeze_rays(rec) as rs:
            rows = rs.status == OK
            rows[:, 0] = False                 # receiver 0: no row
            rows[1:, 1] = False                # receiver 1: one row at most
            assert rows[:, 2:].all()
            b = np.random.default_rng(2).standard_normal(int(rows.sum()))
            h = random_h(b.size, 3)
            for smooth in (0.0, 1.0):
                want = lsqr_joint_restated(*set_operator(rs, rows), b, h, receivers_of(rows), R, dims, damp=1.0,
                                           smooth=smooth, iter_lim=6)
                got = rs.lsqr(b, rows, hypo=h, damp=1.0, smooth=smooth, iter_lim=6)
                assert_same_joint(got, want, f"{dims} {total} smooth {smooth}")
                assert (_bits(got.hypo[0]) == 0).all()


@gpu
def test_joint_lsqr_refusals_leave_the_set_working_and_free_the_workspace():
    ms, rays, rows, b = _golden_problem("rand_818")
    h = random_h(b.size, 8)
    ctx, rs = _golden_set("rand_818")
    with ctx, rs:
        want = rs.lsqr(b, rows, hypo=h, damp=1.0, smooth=1.0, iter_lim=5)
        torch.cuda.synchronize()
        free0 = torch.cuda.mem_get_info()[0]
        for bad, idx in [(np.nan, 13), (np.inf, 0), (-np.inf, 4 * b.size - 1)]:
            hb = h.copy()
            hb.ravel()[idx] = bad
            with pytest.raises(P.SweepError, match=rf"h\[{idx}\] is not finite"):
                rs.lsqr(b, rows, hypo=hb)
        with ctx.freeze_rays(all_nodes(tuple(ms[0]["dims"])), max_nodes=3) as short:
            sel = short.status != OK
            with pytest.raises(P.SweepError, match="not OK"):
                short.lsqr(np.ones(int(sel.sum())), sel, hypo=np.zeros((int(sel.sum()), 4)))
        with pytest.raises(P.SweepError, match="hypo of shape"):
            rs.lsqr(b, rows, hypo=h[:-1])
        with pytest.raises(P.SweepError, match="overflows"):
            bb = b.copy()
            bb[0] = 2.0 ** 600
            rs.lsqr(bb, rows, hypo=h)
        lib = api.load_library()
        x = np.empty(rs.dims, np.float64)
        y = np.empty((rs.shape[1], 4), np.float64)
        sel = np.ascontiguousarray(rows, np.uint8)
        good = api._LsqrOpts(api.C.sizeof(api._LsqrOpts), 1.0, 1.0, 1e-6, 1e-6, 1e8, 5)
        for opts, info in [(api._LsqrOpts(8, 1.0, 1.0, 1e-6, 1e-6, 1e8, 5), None), (good, api._LsqrInfo(4))]:
            assert not lib.sweeptt_rayset_lsqr_hypo(rs._h, sel.ctypes.data, b.ctypes.data, h.ctypes.data,
                                                    api.C.byref(opts), x.ctypes.data, y.ctypes.data,
                                                    api.C.byref(info) if info else None, None)
            assert "struct_size" in lib.sweeptt_last_error().decode()
        for hp, yp in [(None, y.ctypes.data), (h.ctypes.data, None)]:
            assert not lib.sweeptt_rayset_lsqr_hypo(rs._h, sel.ctypes.data, b.ctypes.data, hp, api.C.byref(good),
                                                    x.ctypes.data, yp, None, None)
            assert "hypo_out are required" in lib.sweeptt_last_error().decode()
        torch.cuda.synchronize()
        assert torch.cuda.mem_get_info()[0] == free0
        after = rs.lsqr(b, rows, hypo=h, damp=1.0, smooth=1.0, iter_lim=5)
        assert_same_joint(after, (want.x.ravel(), want.istop, want.itn, want.r1norm, want.r2norm, want.anorm,
                                  want.acond, want.arnorm, want.xnorm, want.hypo), "after the refusals")
        torch.cuda.synchronize()
        assert torch.cuda.mem_get_info()[0] == free0


@gpu
def test_hypocentre_partials_equal_the_rule_on_the_fields():
    """Every node of a box with +inf walls (test_tomography's maze) and of a golden box, faces and edges included."""
    from test_tomography import _maze
    for v, starts in [(_maze(), [(0, 0, 0), (8, 8, 0)]),
                      (W.heterogeneous_field((12, 11, 9), 5), [(0, 0, 0), (11, 10, 8), (5, 5, 4)])]:
        with P.SweepContext() as ctx:
            ctx.set_model(v); ctx.set_star(W.star("818")); ctx.set_sources(starts)
            ctx.run()
            fields = np.stack([ctx.get_tt(s) for s in range(len(starts))])
            centres = all_nodes(v.shape)
            got = P.hypocentre_partials(ctx, centres)
            assert np.array_equal(got, partials_rule(fields, centres), equal_nan=True)
            assert np.isinf(fields).any() == bool(np.isnan(got).any())
            one = P.hypocentre_partials(ctx, centres[:5], sources=(1, 1))
            assert np.array_equal(one, got[:5, 1:2], equal_nan=True)


def _joint_problem(n_events=12, seed=4):
    v = W.heterogeneous_field((33, 25, 40), seed)
    stations = [(0, 0, 0), (32, 24, 0), (0, 24, 39), (32, 0, 39), (16, 12, 0), (16, 0, 20)]
    rng = np.random.default_rng(seed)
    true = np.stack([rng.integers(4, d - 4, n_events) for d in v.shape], axis=1)
    with P.SweepContext() as ctx:
        ctx.set_model((v * rng.uniform(0.98, 1.02, v.shape)).astype(np.float32))
        ctx.set_star(W.star("818")); ctx.set_sources(stations)
        ctx.run()
        t = np.stack([ctx.get_tt(s)[tuple(true.T)] for s in range(len(stations))], axis=1)
    picks = (t + rng.uniform(0, 20, (n_events, 1)) + rng.normal(0, 0.05, t.shape)).astype(np.float32)
    picks[rng.random(picks.shape) < 0.1] = np.nan
    picks[3] = np.nan                                  # an event with no picks: not located
    return v, stations, picks


@gpu
@pytest.mark.parametrize("given", [False, True])
def test_joint_update_equals_its_composition(given):
    v, stations, picks = _joint_problem()
    kw = dict(damp=2.0, smooth=1.0, iter_lim=20)
    with P.SweepContext() as ctx:
        ctx.set_model(v); ctx.set_star(W.star("818")); ctx.set_sources(stations)
        ctx.run()
        loc = ctx.locate_events(picks)
        ok = loc.status == api.LOC_OK
        assert not ok[3] and ok.sum() >= 10
        c = loc.node.copy()
        if given:
            c = np.clip(c + np.array([1, -1, 0]), 0, np.array(v.shape) - 1)
        c = np.where(ok[:, None], c, 0).astype(np.int32)
        with ctx.freeze_rays(c) as rs:
            obs = picks.T.astype(np.float64)
            with np.errstate(invalid="ignore"):
                b = (obs - loc.origin_time) - rs.tt.astype(np.float64)
            rows = np.isfinite(obs) & (rs.status == OK) & ok
            d = P.hypocentre_partials(ctx, c).transpose(1, 0, 2)[rows]
            h = np.concatenate([0.5 * d, np.full((len(d), 1), 3.0)], axis=1)
            want = rs.lsqr(b[rows], rows, hypo=h, **kw)
    got = P.joint_update(v, W.star("818"), stations, picks, centres=c if given else None, hypo_scale=0.5,
                         origin_scale=3.0, **kw)
    assert np.array_equal(got.rows, rows)
    assert (_bits(got.residual[rows]) == _bits(b[rows])).all() and np.isnan(got.residual[~rows]).all()
    assert np.array_equal(got.delta.view(np.uint32), want.x.astype(np.float32).view(np.uint32))
    assert (_bits(got.shift) == _bits(0.5 * want.hypo[:, :3])).all()
    assert (_bits(got.origin_shift) == _bits(3.0 * want.hypo[:, 3])).all()
    assert (got.shift[3] == 0).all() and got.origin_shift[3] == 0 and (got.centres[3] == -1).all()
    assert np.array_equal(got.centres[ok], c[ok])
    assert (got.istop, got.itn, got.r2norm, got.xnorm) == (want.istop, want.itn, want.r2norm, want.xnorm)


@gpu
def test_displaced_events_are_moved_back_on_the_device():
    v = W.constant_field(DISP_DIMS, 0.25)
    centres, true = _disp_events()
    with P.SweepContext() as ctx:
        ctx.set_model(v); ctx.set_star(W.star("818")); ctx.set_sources(DISP_STATIONS)
        ctx.run()
        t = np.stack([ctx.get_tt(s)[DISP_TRUE] for s in range(len(DISP_STATIONS))])
    picks = np.tile(t, (len(centres), 1)).astype(np.float32)
    got = P.joint_update(v, W.star("818"), DISP_STATIONS, picks, centres=centres, damp=DISP_DAMP,
                         iter_lim=DISP_ITERS)
    assert got.rows.all() and (np.abs(got.origin_time) <= 1e-6).all()
    _check_disp(got.shift, true)


@gpu
def test_full_size_config2_joint_lsqr_equals_the_restatement():
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
            h = np.random.default_rng(6).standard_normal((b.size, 4))
            rs.lsqr(b, hypo=h, damp=1.0, smooth=1.0, iter_lim=1)
            torch.cuda.synchronize()
            free0 = torch.cuda.mem_get_info()[0]
            got = rs.lsqr(b, hypo=h, damp=1.0, smooth=1.0, atol=0.0, btol=0.0, iter_lim=4)
            free1 = torch.cuda.mem_get_info()[0]
            want = lsqr_joint_restated(*set_operator(rs, rows), b, h, receivers_of(rows), rows.shape[1], v.shape,
                                       damp=1.0, smooth=1.0, atol=0.0, btol=0.0, iter_lim=4)
            assert_same_joint(got, want, "config 2")
            assert got.itn == 4 and got.istop == 7
    assert free1 == free0, (free0, free1)
