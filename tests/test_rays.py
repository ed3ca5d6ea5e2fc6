"""Rays: shortest paths from receivers back to the start, read off a converged field (include/sweeptt.h,
sweeptt_trace_rays).  CPU: the oracle's rays on every reference-produced golden field end at the start and replay
the field bit for bit; each non-OK status on a built input; the trace kernel never fuses a multiply-add; a C client
links.  GPU (-m gpu): device rays equal oracle rays exactly (nodes, lengths, statuses, receiver times) on every node
of every golden field, whatever kernel or axis permutation produced the field, and on the full-size configs 1 and 2."""
import atexit
import ctypes as C
import functools
import hashlib
import json
import re
import shutil
import subprocess
import tempfile

import numpy as np
import pytest
import torch

import oracle
import uoparallel_seismic_project_b200 as P
from uoparallel_seismic_project_b200 import api, workloads as W

from conftest import ROOT, make_field

gpu = pytest.mark.gpu
OK, UNREACHED, NOT_FIXED, NO_PRED, STALLED, TRUNCATED = range(6)


def all_nodes(dims):
    return np.argwhere(np.ones(tuple(dims), bool)).astype(np.int32)


def half_distance(step, delta=10.0):
    """hd = 0.5f * d of the edge with offsets step[..., 3], d computed the reference's way (make_star)."""
    norm = (step.astype(np.int64) ** 2).sum(-1)
    d = np.float32(delta) * np.sqrt(norm.astype(np.float64)).astype(np.float32)
    return np.float32(0.5) * d


def replay(v, nodes, length, start):
    """Travel times rebuilt along every ray from 0 at the start: t_n = fl(fl(hd * fl(v_n + v_m)) + t_m), m the next
    node.  Returns float32[R, L] (NaN past the length)."""
    nodes = nodes.astype(np.int64)
    R, L = nodes.shape[:2]
    out = np.full((R, L), np.nan, np.float32)
    last = length - 1
    rows = np.arange(R)
    assert (nodes[rows, last] == np.asarray(start)).all(), "a ray does not end at the start"
    t = np.zeros(R, np.float32)
    out[rows, last] = t
    for back in range(1, int(length.max())):
        live = last - back >= 0
        k = np.where(live, last - back, 0)
        n, m = nodes[rows, k], nodes[rows, k + 1]
        vn = v[n[:, 0], n[:, 1], n[:, 2]]
        vm = v[m[:, 0], m[:, 1], m[:, 2]]
        t = np.where(live, half_distance(m - n) * (vn + vm) + t, t).astype(np.float32)
        out[rows[live], k[live]] = t[live]
    return out


def assert_replays(v, tt, nodes, length, start, what=""):
    rep = replay(v, nodes, length, start)
    mask = np.arange(nodes.shape[1])[None, :] < length[:, None]
    idx = nodes[mask].astype(np.int64)
    want = tt[idx[:, 0], idx[:, 1], idx[:, 2]]
    nd = int((rep[mask].view(np.uint32) != want.view(np.uint32)).sum())
    assert nd == 0, f"{what}: {nd} of {mask.sum()} replayed travel times differ from the field"


@functools.lru_cache(maxsize=None)
def _ray_oracle():
    """tests/native/ray_oracle.c built into a temporary directory (the tree may be read-only)."""
    tmp = tempfile.mkdtemp(prefix="ray_oracle_")
    atexit.register(shutil.rmtree, tmp, True)
    so = f"{tmp}/libray_oracle.so"
    subprocess.run(["gcc", "-O3", "-ffp-contract=off", "-fPIC", "-std=gnu11", "-Wall", "-Werror", "-shared", "-o", so,
                    str(ROOT / "tests" / "native" / "ray_oracle.c"), "-lm"], check=True)
    return C.CDLL(so)


def oracle_rays(v, tt, offsets, start, receivers, delta=10.0, used=None, max_nodes=None):
    """CPU rays from every receiver back to `start` through `tt` (tests/native/ray_oracle.c).  Returns
    (nodes int32[R, max_nodes, 3], length int32[R], status int32[R], tt float32[R]); nodes past a length are -1."""
    off = np.ascontiguousarray(offsets, np.int32).reshape(-1, 3)
    used = len(off) - 1 if used is None else used
    v = np.ascontiguousarray(v, np.float32)
    tt = np.ascontiguousarray(tt, np.float32)
    nx, ny, nz = v.shape
    max_nodes = nx + ny + nz if max_nodes is None else max_nodes
    rec = np.ascontiguousarray(receivers, np.int32).reshape(-1, 3)
    nodes = np.full((len(rec), max_nodes, 3), -1, np.int32)
    length, status = np.zeros(len(rec), np.int32), np.zeros(len(rec), np.int32)
    ttr = np.zeros(len(rec), np.float32)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    _ray_oracle().ray_oracle_trace_many(p(v), p(tt), nx, ny, nz, p(off), int(used), C.c_float(delta), int(start[0]),
                                        int(start[1]), int(start[2]), p(rec), len(rec), int(max_nodes), p(nodes),
                                        p(length), p(status), p(ttr))
    return nodes, length, status, ttr


def oracle_ray(v, tt, offsets, start, receiver, delta=10.0, used=None, max_nodes=None):
    """One CPU ray: (nodes int32[L, 3], status, tt[receiver])."""
    nodes, length, status, ttr = oracle_rays(v, tt, offsets, start, [receiver], delta, used, max_nodes)
    return nodes[0, : length[0]].copy(), int(status[0]), ttr[0]


@functools.lru_cache(maxsize=None)
def _golden_cases():
    z = np.load(ROOT / "tests" / "golden" / "small_cases.npz")
    meta = json.loads(bytes(z["meta_json"]).decode())
    by_case = {}
    for m in meta:
        m = dict(m, tt=z[f"{m['case']}__{m['idx']}"])
        by_case.setdefault(m["case"], []).append(m)
    return by_case


@functools.lru_cache(maxsize=None)
def _oracle_rays(case):
    """Oracle rays from every node for every source of a golden case (cached across tests)."""
    ms = _golden_cases()[case]
    v = make_field(ms[0]["kind"], ms[0]["dims"], ms[0]["seed"])
    rec = all_nodes(ms[0]["dims"])
    return [oracle_rays(v, m["tt"], W.star(m["star"]), m["start"], rec) for m in ms]


# ---- CPU: the oracle ---------------------------------------------------------------------------

def test_oracle_rays_from_every_golden_node_reach_the_start_and_replay(golden_small):
    ties = []
    for case, ms in _golden_cases().items():
        v = make_field(ms[0]["kind"], ms[0]["dims"], ms[0]["seed"])
        for m, (nodes, length, status, ttr) in zip(ms, _oracle_rays(case)):
            what = f"{case}[{m['idx']}]"
            assert (status == OK).all(), f"{what}: {np.bincount(status)}"
            assert (ttr == m["tt"].ravel()).all()
            assert_replays(v, m["tt"], nodes, length, m["start"], what)
            if case == "contrast_5fs":
                ties.append(_exact_ties(v, m["tt"], W.star(m["star"]), m["start"]))
    assert ties == [347, 423], "nodes whose best exact matches share tt[m] (the tie rule's second key decides)"


def _exact_ties(v, tt, offsets, start):
    """Nodes at which the exact matches with the smallest tt[m] are not unique (numpy restatement of the edge rules)."""
    off = np.asarray(offsets)[:-1]
    dims = np.array(v.shape)
    nodes = all_nodes(v.shape)
    edges = []   # (node index, index of m, tt[m]) of every exact match
    for sgn in (1, -1):
        for o, dl in zip(off, oracle.star_distances(off)):
            m = nodes + sgn * o
            ok = ((m >= 0) & (m < dims)).all(1) & bool(o.any())
            if sgn < 0:
                ok &= ~(m == np.asarray(start)).all(1)
            n_, m_ = nodes[ok], m[ok]
            tm = tt[tuple(m_.T)]
            cand = ((dl * (v[tuple(n_.T)] + v[tuple(m_.T)])).astype(np.float64) / 2.0).astype(np.float32) + tm
            hit = cand == tt[tuple(n_.T)]
            edges.append((np.nonzero(ok)[0][hit], np.ravel_multi_index(tuple(m_[hit].T), v.shape), tm[hit]))
    i, m, tm = (np.concatenate([e[k] for e in edges]) for k in range(3))
    best = np.full(len(nodes), np.inf, np.float32)
    np.minimum.at(best, i, tm)
    at_best = np.unique(np.stack([i, m])[:, tm == best[i]], axis=1)[0]   # distinct (n, m) pairs
    return int((np.bincount(at_best, minlength=len(nodes)) > 1).sum())


def _status_inputs():
    """(name, v, tt, start, receiver, max_nodes, expected status) built from a golden case."""
    m = _golden_cases()["hetero_818"][0]
    v = make_field(m["kind"], m["dims"], m["seed"])
    star = W.star(m["star"])
    start = tuple(m["start"])
    nodes, length, _, _ = _oracle_rays("hetero_818")[0]
    r = int(np.argmax(length))                      # the longest ray of the field
    path = nodes[r, : length[r]]
    mid = tuple(int(c) for c in path[len(path) // 2])
    out = [("ok", v, m["tt"], start, tuple(path[0]), None, OK),
           ("receiver_is_start", v, m["tt"], start, start, None, OK),
           ("truncated", v, m["tt"], start, tuple(path[0]), 2, TRUNCATED)]
    raised = m["tt"].copy(); raised[mid] = raised[mid] * np.float32(1.5)
    out.append(("raised", v, raised, start, mid, None, NOT_FIXED))
    lowered = m["tt"].copy(); lowered[mid] = lowered[mid] * np.float32(0.5)
    out.append(("lowered", v, lowered, start, mid, None, NO_PRED))
    vinf = v.copy(); vinf[mid] = np.inf
    tinf, _, _ = oracle.solve(vinf, star, start)
    out.append(("inf_slowness", vinf, tinf, start, mid, None, UNREACHED))
    vzero = np.zeros_like(v)
    tzero, _, _ = oracle.solve(vzero, star, start)
    out.append(("zero_model", vzero, tzero, start, tuple(path[0]), None, STALLED))
    return star, out


def test_oracle_statuses_on_built_inputs():
    star, cases = _status_inputs()
    for name, v, tt, start, rec, max_nodes, want in cases:
        nodes, status, ttr = oracle_ray(v, tt, star, start, rec, max_nodes=max_nodes)
        assert status == want, (name, status)
        assert tuple(nodes[0]) == tuple(rec) and ttr.view(np.uint32) == tt[rec].view(np.uint32), name
        if name == "truncated":
            assert len(nodes) == 2
        if name in ("raised", "lowered", "inf_slowness", "zero_model", "receiver_is_start"):
            assert len(nodes) == 1, name


def test_oracle_ray_of_an_unconverged_field_is_flagged():
    m = _golden_cases()["rand_818"][0]
    v = make_field(m["kind"], m["dims"], m["seed"])
    tt = oracle.init_tt(v.shape, m["start"])
    oracle.sweep(v, tt, W.star("818"), m["start"])   # one sweep: not a fixed point yet
    _, _, status, _ = oracle_rays(v, tt, W.star("818"), m["start"], all_nodes(v.shape))
    assert (status == NOT_FIXED).any()


# ---- CPU: the shipped library ------------------------------------------------------------------

@pytest.mark.skipif(shutil.which("cuobjdump") is None, reason="cuobjdump not on PATH")
def test_trace_kernel_never_fuses_multiply_add():
    out = subprocess.run(["cuobjdump", "-sass", str(P.lib_path())], capture_output=True, text=True, check=True).stdout
    funcs, name = {}, None
    for line in out.splitlines():
        mm = re.search(r"Function : (\S+)", line)
        if mm:
            name = mm.group(1)
            funcs[name] = []
        elif name and re.match(r"\s+/\*[0-9a-f]{4,6}\*/", line):
            funcs[name].append(line)
    trace = {k: v for k, v in funcs.items() if "trace_rays" in k}
    assert trace, "no trace_rays kernel in the library"
    for k, lines in trace.items():
        text = "\n".join(lines)
        assert "FMUL" in text and "FADD" in text, k
        assert not re.search(r"\bFFMA2?\b", text), f"{k}: fused multiply-add found"


def test_c99_client_calls_trace_rays(tmp_path):
    """A strict C99 client compiles and links against sweeptt_trace_rays.  Without a GPU the call fails with a
    message; with one it traces a ray through a tiny constant box."""
    src = tmp_path / "client.c"
    src.write_text(r'''
#include <stdio.h>
#include "sweeptt.h"
int main(void) {
  /* symmetric: with one-sided offsets no node could pull from the start (its own visits are skipped) */
  struct FS fs[7] = {{1, 0, 0, 0.f}, {-1, 0, 0, 0.f}, {0, 1, 0, 0.f}, {0, -1, 0, 0.f}, {0, 0, 1, 0.f},
                     {0, 0, -1, 0.f}, {1, 1, 1, 0.f}};
  struct START st[1] = {{0, 0, 0}}, rec[2] = {{3, 3, 3}, {0, 0, 0}}, nodes[2 * 16];
  float v[64], tt[2];
  int32_t len[2], status[2];
  sweeptt_stats stats;
  sweeptt_ctx *ctx;
  int i;
  for (i = 0; i < 64; i++) v[i] = 1.f;
  sweeptt_star_fill_distances(fs, 7, 10.0f);
  ctx = sweeptt_create(NULL);
  if (!ctx) {
    if (sweeptt_trace_rays(NULL, 0, 1, rec, 2, 16, nodes, len, status, tt, &stats)) return 2;
    printf("%s\n", sweeptt_last_error());
    return 0;
  }
  if (!sweeptt_set_model(ctx, v, 4, 4, 4) || !sweeptt_set_star(ctx, fs, 7) || !sweeptt_set_sources(ctx, st, 1) ||
      !sweeptt_run(ctx, NULL) || !sweeptt_trace_rays(ctx, 0, 1, rec, 2, 16, nodes, len, status, tt, &stats)) {
    printf("%s\n", sweeptt_last_error());
    return 3;
  }
  sweeptt_destroy(ctx);
  if (status[0] != SWEEPTT_RAY_OK || len[0] != 10 || status[1] != SWEEPTT_RAY_OK || len[1] != 1) return 4;
  if (nodes[9].i != 0 || nodes[9].j != 0 || nodes[9].k != 0 || tt[0] != 90.f) return 5;
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
    assert ("ok" if torch.cuda.is_available() else "null context") in r.stdout


# ---- GPU ---------------------------------------------------------------------------------------

def _device_rays(ms, kernel=None, put=False, max_nodes=None):
    v = make_field(ms[0]["kind"], ms[0]["dims"], ms[0]["seed"])
    with P.SweepContext(kernel=kernel) as ctx:
        ctx.set_model(v); ctx.set_star(W.star(ms[0]["star"])); ctx.set_sources([m["start"] for m in ms])
        if put:
            for s, m in enumerate(ms):
                ctx.put_tt(s, m["tt"])
        else:
            ctx.run()
        return ctx.trace_rays(all_nodes(ms[0]["dims"]), max_nodes=max_nodes)


def _assert_rays_equal(got, want, what):
    """got / want: (nodes [R, L, 3], length [R], status [R], tt [R]) of one source."""
    nodes, length, status, ttr = want
    assert (got[2] == status).all(), f"{what}: statuses differ"
    assert (got[1] == length).all(), f"{what}: lengths differ"
    assert (got[3].view(np.uint32) == ttr.view(np.uint32)).all(), f"{what}: receiver times differ"
    L = min(nodes.shape[1], got[0].shape[1])
    assert (length <= L).all()
    assert (got[0][:, :L] == nodes[:, :L]).all(), f"{what}: nodes differ"


def _one(rays, s, pick=slice(None)):
    return rays.nodes[s, pick], rays.length[s, pick], rays.status[s, pick], rays.tt[s, pick]


def _check_every_golden(**kw):
    for case, ms in _golden_cases().items():
        rays = _device_rays(ms, **kw)
        assert rays.stats.kernel_launches == 1 and rays.stats.relaxations > 0 and rays.stats.solve_ms > 0
        for s, want in enumerate(_oracle_rays(case)):
            _assert_rays_equal(_one(rays, s), want, f"{case}[{s}] {kw}")


@gpu
@pytest.mark.parametrize("kernel", [api.KERNEL_SIMPLE, api.KERNEL_TILED])
def test_device_rays_equal_oracle_on_every_golden_node(kernel):
    _check_every_golden(kernel=kernel)


@gpu
@pytest.mark.parametrize("axis", ["0", "1", "2"])
def test_device_rays_do_not_depend_on_the_axis_permutation(axis, monkeypatch):
    monkeypatch.setenv("SWEEPTT_WINDOW_AXIS", axis)
    _check_every_golden()


@gpu
def test_device_rays_of_fields_loaded_with_put_tt():
    _check_every_golden(put=True)


@gpu
def test_device_statuses_equal_oracle():
    star, cases = _status_inputs()
    for name, v, tt, start, rec, max_nodes, want in cases:
        with P.SweepContext() as ctx:
            ctx.set_model(v); ctx.set_star(star); ctx.set_sources([start]); ctx.put_tt(0, tt)
            rays = ctx.trace_rays([rec], max_nodes=max_nodes)
        o = oracle_rays(v, tt, star, start, [rec], max_nodes=max_nodes)
        assert rays.status[0, 0] == want, (name, rays.status[0, 0])
        _assert_rays_equal(_one(rays, 0), o, name)


@gpu
def test_device_unreached_and_stalled_after_a_solve():
    star, cases = _status_inputs()
    for name, v, tt, start, rec, _, want in cases:
        if name not in ("inf_slowness", "zero_model"):
            continue
        rays = P.trace_rays(v, star, [start], [rec])
        assert rays.status[0, 0] == want and rays.tt[0, 0].view(np.uint32) == tt[rec].view(np.uint32), name


@gpu
def test_star_wider_than_the_tiled_halo():
    """|i| = 9 does not fit the tiled kernel's halo: the field comes from the simple kernel, the rays from the same
    tracer."""
    off = np.concatenate([W.star("5")[:-1], [[9, 1, 0], [-9, 0, 2], [0, 0, 0]]]).astype(np.int32)
    v = W.random_field((22, 13, 11), seed=12)
    starts = [(3, 6, 5), (21, 0, 10)]
    rec = all_nodes(v.shape)
    with P.SweepContext() as ctx:
        ctx.set_model(v); ctx.set_star(off); ctx.set_sources(starts)
        st = ctx.run()
        assert st.kernel_used == api.KERNEL_SIMPLE
        rays = ctx.trace_rays(rec)
    for s, p in enumerate(starts):
        tt, _, _ = oracle.solve(v, off, p)
        want = oracle_rays(v, tt, off, p, rec)
        assert (want[2] == OK).all()
        _assert_rays_equal(_one(rays, s), want, f"source {s}")
        x = want[0][..., 0]
        assert ((np.abs(np.diff(x, axis=1)) == 9) & (x[:, 1:] >= 0) & (x[:, :-1] >= 0)).any(), "no |i| = 9 step"


@gpu
def test_source_range_slicing_matches_one_full_call():
    ms = _golden_cases()["hetero_818"]
    v = make_field(ms[0]["kind"], ms[0]["dims"], ms[0]["seed"])
    rec = all_nodes(v.shape)[::7]
    with P.SweepContext() as ctx:
        ctx.set_model(v); ctx.set_star(W.star("818")); ctx.set_sources([m["start"] for m in ms])
        ctx.run()
        full = ctx.trace_rays(rec)
        parts = [ctx.trace_rays(rec, sources=range(s, s + 1), max_nodes=full.nodes.shape[2]) for s in range(3)]
        tail = ctx.trace_rays(rec, sources=(1, 2), max_nodes=full.nodes.shape[2])
        with pytest.raises(P.SweepError, match="not within"):
            ctx.trace_rays(rec, sources=(2, 2))
        with pytest.raises(P.SweepError, match="outside"):
            ctx.trace_rays([(0, 0, 40)])
        with pytest.raises(P.SweepError, match="max_nodes"):
            ctx.trace_rays(rec, max_nodes=0)
    for s, part in enumerate(parts):
        for f in ("tt", "status", "length", "nodes"):
            assert (getattr(part, f)[0] == getattr(full, f)[s]).all(), (s, f)
    for f in ("tt", "status", "length", "nodes"):
        assert (getattr(tail, f) == getattr(full, f)[1:]).all(), f


def _full_size(label, v, star, kernel):
    gold = [g for g in json.loads((ROOT / "tests" / "golden" / "full_241.json").read_text()) if g["label"].startswith(label)]
    assert hashlib.sha256(v.tobytes()).hexdigest() == gold[0]["v_sha256"]
    starts = [g["start"] for g in gold]
    face = np.array([(x, y, 0) for x in range(241) for y in range(241)], np.int32)   # the z = 0 face: 58,081 nodes
    rng = np.random.default_rng(2024)
    with P.SweepContext(kernel=kernel) as ctx:
        ctx.set_model(v); ctx.set_star(star); ctx.set_sources(starts)
        ctx.run()
        fields = [ctx.get_tt(s) for s in range(len(starts))]
        rays = ctx.trace_rays(face)
    for s, (g, tt) in enumerate(zip(gold, fields)):
        assert hashlib.sha256(tt.tobytes()).hexdigest() == g["tt_sha256"], f"{g['label']}: field differs"
        assert (rays.status[s] == OK).all(), np.bincount(rays.status[s])
        assert (rays.tt[s] == tt[:, :, 0].ravel()).all()
        assert_replays(v, tt, rays.nodes[s], rays.length[s], g["start"], g["label"])
        pick = rng.choice(len(face), 200, replace=False)
        want = oracle_rays(v, tt, star, g["start"], face[pick], max_nodes=rays.nodes.shape[2])
        _assert_rays_equal(_one(rays, s, pick), want, g["label"])


@gpu
def test_full_size_config1_constant_3fs_face_rays():
    _full_size("config1", W.constant_field((241, 241, 51)), W.star("3"), None)


@gpu
def test_full_size_config2_heterogeneous_818_face_rays():
    _full_size("config2", W.heterogeneous_field((241, 241, 51), seed=7), W.star("818"), api.KERNEL_TILED)
