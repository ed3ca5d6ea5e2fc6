"""Ray sets: rays traced once and kept on the device (include/sweeptt.h, sweeptt_rayset_*), and the damped LSQR step.

The yardsticks are the operators of test_tomography.py (ray_project / ray_backproject and their oracles) and the rays
of test_rays.py: a set's table, paths and operators must equal them bit for bit.  CPU: the new kernels never fuse a
multiply-add; a C99 client links against every entry point; the LSQR reference (scipy's lsqr on the oracle operators,
with the documented float32 conversions) agrees with lsqr on the explicit float64 G within a bound derived from the
condition number.  GPU (-m gpu): every golden node under both kernels, every axis permutation and put_tt; snapshot
semantics; rays that are not OK; truncation and the default retry; determinism; memory; closing; full-size config 2;
linearized_update bit for bit against the LSQR reference."""
import hashlib
import json
import re
import shutil
import subprocess

import numpy as np
import pytest
import torch
from scipy.sparse.linalg import LinearOperator, lsqr

import oracle
import uoparallel_seismic_project_b200 as P
from uoparallel_seismic_project_b200 import api, workloads as W

from conftest import ROOT, make_field
from test_rays import _golden_cases, _oracle_rays, all_nodes, half_distance, oracle_rays
from test_tomography import (AXIS_STAR, _bits_equal, _ctx, _edges, _hd_max, _maze, _weights, oracle_backproject,
                             oracle_project)

gpu = pytest.mark.gpu
OK, TRUNCATED = api.RAY_OK, api.RAY_TRUNCATED
U = 2.0 ** -24   # unit roundoff of float32


# ---- the LSQR reference ------------------------------------------------------------------------

def _case_problem(case, seed=6):
    """Oracle rays of every node of a golden case, its receiver times and 'observed' times 3 % off (seeded)."""
    ms = _golden_cases()[case]
    rays = [r[:3] for r in _oracle_rays(case)]
    t = np.stack([m["tt"].ravel() for m in ms])
    obs = (t * np.random.default_rng(seed).uniform(0.97, 1.03, t.shape)).astype(np.float32)
    return ms, rays, t, obs


def oracle_operator(dims, rays, rows, hd_max):
    """G over the rays selected by rows [S, R] from the CPU oracles, with RaySet.as_linear_operator's conversions."""
    S, R = rows.shape

    def matvec(x):
        d = np.asarray(x, np.float32).reshape(dims)
        return np.stack([oracle_project(d, *r) for r in rays])[rows].astype(np.float64)

    def rmatvec(y):
        w = np.zeros((S, R), np.float32)
        w[rows] = np.asarray(y, np.float32).ravel()
        return oracle_backproject(dims, rays, w, hd_max)[0].astype(np.float64).ravel()

    return LinearOperator((int(rows.sum()), int(np.prod(dims))), matvec=matvec, rmatvec=rmatvec, dtype=np.float64)


def lsqr_reference(case, damp, iter_lim, atol=1e-6, btol=1e-6):
    """linearized_update restated on the CPU: r = float32(observed - t) over the OK rays with a pick, then scipy's lsqr
    on the oracle operator.  Returns (delta float32[dims], residual [S, R], lsqr's tuple)."""
    ms, rays, t, obs = _case_problem(case)
    dims = tuple(ms[0]["dims"])
    status = np.stack([r[2] for r in rays])
    residual = (obs - t).astype(np.float32)
    use = np.isfinite(residual) & (status == OK)
    residual = np.where(use, residual, np.float32(np.nan)).astype(np.float32)
    op = oracle_operator(dims, rays, use, _hd_max(ms[0]["star"]))
    out = lsqr(op, residual[use].astype(np.float64), damp=damp, atol=atol, btol=btol, iter_lim=iter_lim)
    return out[0].astype(np.float32).reshape(dims), residual, out


def explicit_g(dims, rays, rows):
    """The float64 matrix G of the rays selected by rows: hd of every edge at both of its ends."""
    G = np.zeros(rows.shape + (int(np.prod(dims)),))
    for s, (nodes, length, _) in enumerate(rays):
        for live, n, m in _edges(nodes, length):
            q = np.nonzero(live)[0]
            hd = half_distance(m[q] - n[q]).astype(np.float64)
            np.add.at(G[s], (q, np.ravel_multi_index(tuple(n[q].T), dims)), hd)
            np.add.at(G[s], (q, np.ravel_multi_index(tuple(m[q].T), dims)), hd)
    return G[rows]


# ---- CPU ---------------------------------------------------------------------------------------

def test_lsqr_reference_agrees_with_lsqr_on_the_explicit_matrix():
    """Both runs converge (atol = btol = 1e-10) on the damped system A = [G; damp I].  The float32 operators apply A
    exactly up to a relative perturbation eps = (L_max + 2) u per entry: the (L + 1) u of a ray's float32 path sum
    (test_tomography's adjoint bound), plus the float32 rounding of x or y.  The perturbation bound of least squares
    (Golub & Van Loan, Thm. 5.3.1) then gives |dx|/|x| <= eps kappa (2 + kappa |res| / (|A| |x|)), kappa the condition
    number of A from a dense SVD, res the exact residual."""
    damp = 20.0
    delta, residual, out = lsqr_reference("rand_818", damp, 400, atol=1e-10, btol=1e-10)
    ms, rays, _, _ = _case_problem("rand_818")
    dims = tuple(ms[0]["dims"])
    use = np.isfinite(residual)
    G = explicit_g(dims, rays, use)
    b = residual[use].astype(np.float64)
    ref = lsqr(G, b, damp=damp, atol=1e-10, btol=1e-10, iter_lim=400)
    assert out[1] in (1, 2) and ref[1] in (1, 2), (out[1], ref[1])
    sv = np.linalg.svd(G, compute_uv=False)
    norm_a = np.hypot(sv[0], damp)
    kappa = norm_a / np.hypot(sv[-1], damp)
    n = G.shape[1]
    A = np.vstack([G, damp * np.eye(n)])
    x = np.linalg.lstsq(A, np.concatenate([b, np.zeros(n)]), rcond=None)[0]
    res = np.linalg.norm(np.concatenate([b, np.zeros(n)]) - A @ x)
    eps = (max(int(r[1].max()) for r in rays) + 2) * U
    tol = eps * kappa * (2 + kappa * res / (norm_a * np.linalg.norm(x)))
    err = np.linalg.norm(delta.astype(np.float64).ravel() - ref[0]) / np.linalg.norm(ref[0])
    assert err <= tol, (err, tol, kappa)


@pytest.mark.skipif(shutil.which("cuobjdump") is None, reason="cuobjdump not on PATH")
def test_rayset_kernels_never_fuse_multiply_add():
    out = subprocess.run(["cuobjdump", "-sass", str(P.lib_path())], capture_output=True, text=True, check=True).stdout
    funcs, name = {}, None
    for line in out.splitlines():
        mm = re.search(r"Function : (\S+)", line)
        if mm:
            name = mm.group(1)
            funcs[name] = []
        elif name and re.match(r"\s+/\*[0-9a-f]{4,6}\*/", line):
            funcs[name].append(line)
    kernels = {k: v for k, v in funcs.items() if "rayset_" in k}
    assert len(kernels) == 4, sorted(kernels)
    for k, lines in kernels.items():
        text = "\n".join(lines)
        if "rayset_project" in k:
            assert "FMUL" in text and "FADD" in text, k
        assert not re.search(r"\bFFMA2?\b", text), f"{k}: fused multiply-add found"


def test_c99_client_calls_every_rayset_entry_point(tmp_path):
    """A strict C99 client compiles and links against every ray-set entry point.  Without a GPU each call fails with a
    message; with one, on a tiny constant box, the projection of the slowness is the receiver's time and paths() is
    the straight ray."""
    src = tmp_path / "client.c"
    src.write_text(r'''
#include <stdio.h>
#include "sweeptt.h"
int main(void) {
  struct FS fs[7] = {{1, 0, 0, 0.f}, {-1, 0, 0, 0.f}, {0, 1, 0, 0.f}, {0, -1, 0, 0.f}, {0, 0, 1, 0.f},
                     {0, 0, -1, 0.f}, {1, 1, 1, 0.f}};
  struct START st[1] = {{0, 0, 0}}, rec[2] = {{3, 0, 0}, {0, 0, 0}}, nodes[8];
  float v[64], proj[2], w[2] = {1.f, 1.f}, grad[64], tt[2];
  int32_t len[2], status[2];
  int64_t off[3];
  int e = -1, i, fails = 0;
  sweeptt_stats stats;
  sweeptt_ctx *ctx;
  sweeptt_rayset *set;
  for (i = 0; i < 64; i++) v[i] = 1.f;
  sweeptt_star_fill_distances(fs, 7, 10.0f);
  ctx = sweeptt_create(NULL);
  if (!ctx) {
    if (sweeptt_rayset_freeze(NULL, 0, 1, rec, 2, 16, &stats)) return 2;
    printf("%s\n", sweeptt_last_error());
    fails += !sweeptt_rayset_table(NULL, len, status, tt);
    fails += !sweeptt_rayset_paths(NULL, off, nodes);
    fails += !sweeptt_rayset_project(NULL, v, proj, &stats);
    fails += !sweeptt_rayset_backproject(NULL, w, grad, &e, &stats);
    printf("%s\n", sweeptt_last_error());
    sweeptt_rayset_destroy(NULL);
    return fails == 4 && sweeptt_rayset_bytes(NULL) == 0 ? 0 : 2;
  }
  if (!sweeptt_set_model(ctx, v, 4, 4, 4) || !sweeptt_set_star(ctx, fs, 7) || !sweeptt_set_sources(ctx, st, 1) ||
      !sweeptt_run(ctx, NULL) || !(set = sweeptt_rayset_freeze(ctx, 0, 1, rec, 2, 16, &stats)) ||
      !sweeptt_rayset_table(set, len, status, tt) || !sweeptt_rayset_paths(set, off, NULL) ||
      !sweeptt_rayset_paths(set, NULL, nodes) || !sweeptt_rayset_project(set, v, proj, &stats) ||
      !sweeptt_rayset_backproject(set, w, grad, &e, &stats)) {
    printf("%s\n", sweeptt_last_error());
    return 3;
  }
  if (sweeptt_rayset_bytes(set) == 0) return 4;
  sweeptt_rayset_destroy(set);
  sweeptt_destroy(ctx);
  if (status[0] != SWEEPTT_RAY_OK || len[0] != 4 || proj[0] != 30.f || proj[1] != 0.f || tt[0] != 30.f) return 5;
  if (off[0] != 0 || off[1] != 4 || off[2] != 5) return 6;
  for (i = 0; i < 4; i++)
    if (nodes[i].i != 3 - i || nodes[i].j != 0 || nodes[i].k != 0) return 7;
  if (nodes[4].i != 0 || grad[0] != 5.f || grad[16] != 10.f || grad[48] != 5.f) return 8;
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
        assert "null context" in r.stdout and "null ray set" in r.stdout, r.stdout


# ---- GPU ---------------------------------------------------------------------------------------

def _assert_set_equals_operators(ctx, rs, rec, d, w, what, rays=None):
    """The set's table, paths and operators against trace_rays / ray_project / ray_backproject of the same context (and
    the oracle rays when given)."""
    tr = ctx.trace_rays(rec)
    assert (rs.status == tr.status).all() and (rs.length == tr.length).all(), what
    assert _bits_equal(rs.tt, tr.tt), what
    offsets, nodes = rs.paths()
    ok = (rs.status == OK).ravel()
    want_len = np.where(ok, rs.length.ravel(), 0)
    assert (np.diff(offsets) == want_len).all() and offsets[0] == 0, what
    want = np.concatenate([tr.nodes.reshape(-1, tr.nodes.shape[2], 3)[q, :want_len[q]] for q in np.nonzero(ok)[0]]
                          or [np.zeros((0, 3), np.int32)])
    assert (nodes == want).all(), f"{what}: paths() differ from trace_rays"
    pd, bp = ctx.ray_project(d, rec), ctx.ray_backproject(w, rec)
    spd, sbp = rs.project(d), rs.backproject(w)
    assert _bits_equal(spd.values, pd.values), f"{what}: projection"
    assert sbp.quantum_exp == bp.quantum_exp and _bits_equal(sbp.grad, bp.grad), f"{what}: back-projection"
    assert spd.stats.kernel_launches == 2 and spd.stats.solve_ms > 0 and sbp.stats.solve_ms > 0
    if rays is not None:
        for s, (nodes_o, length_o, status_o) in enumerate(rays):
            assert _bits_equal(spd.values[s], oracle_project(d, nodes_o, length_o, status_o)), f"{what}: oracle"
    return spd, sbp


def _check_every_golden(**kw):
    for case, ms in _golden_cases().items():
        dims = tuple(ms[0]["dims"])
        rec = all_nodes(dims)
        rays = [r[:3] for r in _oracle_rays(case)]
        ctx, v = _ctx(ms, **kw)
        with ctx:
            d = np.random.default_rng(1).standard_normal(dims).astype(np.float32)
            w = _weights((len(ms), len(rec)), 2)
            with ctx.freeze_rays(rec) as rs:
                assert rs.stats.relaxations > 0 and rs.stats.solve_ms > 0
                _, sbp = _assert_set_equals_operators(ctx, rs, rec, d, w, f"{case} {kw}", rays)
                assert _bits_equal(rs.project(v).values, np.stack([m["tt"].ravel() for m in ms]))
        g, e = oracle_backproject(dims, rays, w, _hd_max(ms[0]["star"]))
        assert sbp.quantum_exp == e and _bits_equal(sbp.grad, g), f"{case} {kw}: oracle back-projection"


@gpu
@pytest.mark.parametrize("kernel", [api.KERNEL_SIMPLE, api.KERNEL_TILED])
def test_rayset_equals_operators_on_every_golden_node(kernel):
    _check_every_golden(kernel=kernel)


@gpu
@pytest.mark.parametrize("axis", ["0", "1", "2"])
def test_rayset_does_not_depend_on_the_axis_permutation(axis, monkeypatch):
    monkeypatch.setenv("SWEEPTT_WINDOW_AXIS", axis)
    _check_every_golden()


@gpu
def test_rayset_of_fields_loaded_with_put_tt():
    _check_every_golden(put=True)


@gpu
def test_rayset_is_a_snapshot():
    """After the freeze the context gets another model (other dimensions), another star, fields from run and put_tt:
    the set still gives the results of the frozen state."""
    ms = _golden_cases()["hetero_818"]
    dims = tuple(ms[0]["dims"])
    rec = all_nodes(dims)[::2]
    d = np.random.default_rng(21).standard_normal(dims).astype(np.float32)
    w = _weights((len(ms), len(rec)), 22)
    ctx, v = _ctx(ms)
    with ctx:
        pd, bp = ctx.ray_project(d, rec), ctx.ray_backproject(w, rec)
        rs = ctx.freeze_rays(rec)
        nbytes, table = rs.nbytes, (rs.status.copy(), rs.length.copy(), rs.tt.copy())
        paths = rs.paths()
        other = _golden_cases()["contrast_5fs"]
        ctx.set_model(make_field(other[0]["kind"], other[0]["dims"], other[0]["seed"]))
        ctx.set_star(W.star(other[0]["star"]))
        ctx.set_sources([m["start"] for m in other])
        ctx.run()
        ctx.put_tt(0, other[0]["tt"])
        spd, sbp = rs.project(d), rs.backproject(w)
        assert _bits_equal(spd.values, pd.values) and sbp.quantum_exp == bp.quantum_exp and _bits_equal(sbp.grad, bp.grad)
        assert rs.nbytes == nbytes and all((a == b).all() for a, b in zip(table, (rs.status, rs.length, rs.tt)))
        again = rs.paths()
        assert (again[0] == paths[0]).all() and (again[1] == paths[1]).all()
        with pytest.raises(P.SweepError, match="shape"):
            rs.project(np.zeros(other[0]["dims"], np.float32))


@gpu
def test_rays_that_are_not_ok_are_nan_and_contribute_nothing():
    ms = _golden_cases()["hetero_818"]
    dims = tuple(ms[0]["dims"])
    rec = all_nodes(dims)
    ctx, v = _ctx(ms, put=True)
    with ctx:
        ctx.reset()
        ctx.step(3)   # not converged: some rays are NOT_FIXED_POINT / NO_PREDECESSOR
        w = np.random.default_rng(4).choice(np.array([1.0, -1.0, 0.5], np.float32), (ctx.nsrc, len(rec)))
        with ctx.freeze_rays(rec) as rs:
            assert (rs.status != OK).any() and (rs.status == OK).any()
            d = np.random.default_rng(5).standard_normal(dims).astype(np.float32)
            spd, _ = _assert_set_equals_operators(ctx, rs, rec, d, w, "unconverged")
            assert np.isnan(spd.values[rs.status != OK]).all() and not np.isnan(spd.values[rs.status == OK]).any()
            full = rs.backproject(w)
            only_ok = rs.backproject(np.where(rs.status == OK, w, np.float32(0)))
            assert full.quantum_exp == only_ok.quantum_exp and _bits_equal(full.grad, only_ok.grad)
            offsets, _ = rs.paths()
            assert (np.diff(offsets)[(rs.status != OK).ravel()] == 0).all()


@gpu
def test_small_max_nodes_truncates_and_the_default_grows():
    ms = _golden_cases()["hetero_818"]
    dims = tuple(ms[0]["dims"])
    rec = all_nodes(dims)[::5]
    ctx, v = _ctx(ms)
    with ctx:
        with ctx.freeze_rays(rec, max_nodes=3) as rs:
            short = ctx.ray_project(v, rec, max_nodes=3)
            assert (rs.status == TRUNCATED).any() and (rs.status == OK).any() and (rs.length <= 3).all()
            assert (rs.status == short.status).all() and _bits_equal(rs.project(v).values, short.values)
        with pytest.raises(P.SweepError, match="max_nodes"):
            ctx.freeze_rays(rec, max_nodes=0)
        with pytest.raises(P.SweepError, match="outside"):
            ctx.freeze_rays([(0, 0, 99)])
        with pytest.raises(P.SweepError, match="not within"):
            ctx.freeze_rays(rec, sources=(2, 2))
    v = _maze()
    start, far = (0, 0, 0), (8, 8, 0)
    tt, _, _ = oracle.solve(v, AXIS_STAR, start)
    nodes, length, status, _ = oracle_rays(v, tt, AXIS_STAR, start, [far], max_nodes=200)
    with P.SweepContext() as ctx:
        ctx.set_model(v); ctx.set_star(AXIS_STAR); ctx.set_sources([start])
        ctx.run()
        with ctx.freeze_rays([far], max_nodes=sum(v.shape)) as cut, ctx.freeze_rays([far]) as grown:
            assert cut.status[0, 0] == TRUNCATED and np.isnan(cut.project(v).values[0, 0])
            assert grown.status[0, 0] == OK and grown.length[0, 0] == length[0] > 2 * sum(v.shape)
            assert _bits_equal(grown.project(v).values[0, 0], tt[far])
            offsets, got = grown.paths()
            assert (got == nodes[0, : length[0]]).all()
            with pytest.raises(P.SweepError, match="not finite"):
                grown.backproject(np.full((1, 1), np.inf, np.float32))


@gpu
def test_rayset_is_deterministic():
    ms = _golden_cases()["hetero_818"]
    dims = tuple(ms[0]["dims"])
    rec = all_nodes(dims)
    w = _weights((len(ms), len(rec)), 8)
    ctx, v = _ctx(ms)
    with ctx:
        with ctx.freeze_rays(rec) as a, ctx.freeze_rays(rec) as b:
            pa, pb = a.paths(), b.paths()
            assert (pa[0] == pb[0]).all() and (pa[1] == pb[1]).all() and a.nbytes == b.nbytes
            g = [a.backproject(w) for _ in range(3)] + [b.backproject(w)]
            assert all(x.quantum_exp == g[0].quantum_exp and _bits_equal(x.grad, g[0].grad) for x in g)


def _bytes_besides_boxes(rs, npull, nsrc):
    """include/sweeptt.h: nbytes = 2 P + 16 N + 8 + 16 npull + 8 S + 12 V + 4 D; all of it but the 12 V of the two padded
    boxes, whose padded volume V the library derives from its tiling."""
    nx, ny, nz = rs.dims
    offsets, _ = rs.paths()
    entries = int(np.where(rs.status == OK, rs.length - 1, 0).sum())
    assert int(offsets[-1]) == entries + int((rs.status == OK).sum())
    return 2 * entries + 16 * rs.status.size + 8 + 16 * npull + 8 * nsrc + 4 * nx * ny * nz


@gpu
def test_rayset_memory_is_reported_and_released():
    """nbytes follows the documented layout (the padded-box terms are the difference of two sets on the same box), it
    is not counted in pool_bytes, and ctx.close() closes every live set: a closed set raises."""
    ms = _golden_cases()["hetero_818"]
    dims = tuple(ms[0]["dims"])
    rec = all_nodes(dims)
    npull = len(P.build_pull_star(W.star("818"))[0])
    ctx, v = _ctx(ms)
    with ctx:
        a = ctx.freeze_rays(rec)
        pool = ctx.pool_bytes
        b = ctx.freeze_rays(rec[:100], sources=(1, 1))
        assert ctx.pool_bytes == pool, "a set's own memory is not the context's pool"
        # both hold two padded boxes of the same V: what is left besides them is the same 12 V
        boxes = a.nbytes - _bytes_besides_boxes(a, npull, 3)
        assert boxes == b.nbytes - _bytes_besides_boxes(b, npull, 1) and boxes % 12 == 0
        assert boxes // 12 >= (dims[0] + 14) * (dims[1] + 14) * (dims[2] + 16)   # the aprons of device_types.h
        b.close()
        with pytest.raises(P.SweepError, match="closed"):
            b.project(v)
    with pytest.raises(P.SweepError, match="closed"):
        a.backproject(np.zeros(a.shape, np.float32))
    with pytest.raises(P.SweepError, match="closed"):
        a.nbytes


@gpu
def test_full_size_config2_rayset_equals_the_operators():
    v = W.heterogeneous_field((241, 241, 51), seed=7)
    star = W.star("818")
    gold = [g for g in json.loads((ROOT / "tests" / "golden" / "full_241.json").read_text())
            if g["label"].startswith("config2")]
    assert hashlib.sha256(v.tobytes()).hexdigest() == gold[0]["v_sha256"]
    starts = [g["start"] for g in gold]
    face = np.array([(x, y, 0) for x in range(241) for y in range(241)], np.int32)
    d = np.random.default_rng(31).standard_normal(v.shape).astype(np.float32)
    w = _weights((len(starts), len(face)), 32)
    with P.SweepContext(kernel=api.KERNEL_TILED) as ctx:
        ctx.set_model(v); ctx.set_star(star); ctx.set_sources(starts)
        ctx.run()
        pd, bp = ctx.ray_project(d, face), ctx.ray_backproject(w, face)
        rs = ctx.freeze_rays(face)
        assert (rs.status == OK).all()
        spd, sbp = rs.project(d), rs.backproject(w)
        assert _bits_equal(spd.values, pd.values)
        assert sbp.quantum_exp == bp.quantum_exp and _bits_equal(sbp.grad, bp.grad)
        assert _bits_equal(rs.project(v).values, rs.tt)
        nbytes = rs.nbytes
        torch.cuda.synchronize()
        free0 = torch.cuda.mem_get_info()[0]
        rs.close()
        free1 = torch.cuda.mem_get_info()[0]
    assert free1 - free0 >= nbytes // 2, (free1 - free0, nbytes)


@gpu
def test_linearized_update_equals_the_lsqr_reference():
    """The GPU step and the CPU restatement run scipy's lsqr on operators that agree bit for bit, so every iterate
    and delta agree bit for bit."""
    damp, iters = 20.0, 25
    want, want_res, out = lsqr_reference("rand_818", damp, iters)
    ms, _, _, obs = _case_problem("rand_818")
    dims = tuple(ms[0]["dims"])
    v = make_field(ms[0]["kind"], dims, ms[0]["seed"])
    got = P.linearized_update(v, W.star(ms[0]["star"]), [m["start"] for m in ms], all_nodes(dims), obs, damp=damp,
                              iter_lim=iters)
    assert _bits_equal(got.residual, want_res)
    assert got.istop == out[1] and got.iterations == out[2] and got.residual_norm == out[3]
    assert _bits_equal(got.delta, want), f"delta differs in {int((got.delta != want).sum())} nodes"
    use = np.isfinite(want_res)
    assert got.misfit == 0.5 * float(np.sum(want_res[use].astype(np.float64) ** 2))


@gpu
def test_linearized_update_lowers_the_linearised_misfit():
    ms, _, t, obs = _case_problem("hetero_818", seed=7)
    dims = tuple(ms[0]["dims"])
    v = make_field(ms[0]["kind"], dims, ms[0]["seed"])
    rec = all_nodes(dims)[::3]
    idx = np.ravel_multi_index(tuple(rec.T), dims)
    obs = obs[:, idx]
    obs[np.random.default_rng(8).random(obs.shape) < 0.1] = np.nan   # no pick
    starts = [m["start"] for m in ms]
    up = P.linearized_update(v, W.star("818"), starts, rec, obs, damp=5.0, iter_lim=30)
    assert up.istop in range(8) and 0 < up.iterations <= 30
    use = np.isfinite(up.residual)
    assert use.sum() == np.isfinite(obs).sum()
    with P.SweepContext() as ctx:
        ctx.set_model(v); ctx.set_star(W.star("818")); ctx.set_sources(starts); ctx.run()
        with ctx.freeze_rays(rec) as rs:
            gd = rs.project(up.delta).values
    after = 0.5 * float(np.sum((up.residual[use].astype(np.float64) - gd[use]) ** 2))
    assert after < up.misfit, (after, up.misfit)
    assert abs(np.sqrt(2 * after) - up.residual_norm) <= 1e-2 * up.residual_norm
