#!/usr/bin/env python3
"""rayset_bench.py -- rays frozen once as a ray set, then G*d and G^T*w from the stored rays, on one GPU.

  python tools/rayset_bench.py [--workload config3|config2] [--chunk S] [--reps K] [--lsqr-iters N] [--out FILE]

The workloads of tools/tomo_bench.py: the 241x241x51 heterogeneous box (seed 7), 818-FS, config 3 = 111 starts,
config 2 = 4, solved device-resident; "observed" receiver times from a second context on the model perturbed by
U(0.98, 1.02) (seed 8); every receiver of the face z = 0 (58,081 per source).  In one process it measures:
  - the freeze of every ray (device time from the call's stats, and the host wall clock) and the set's nbytes;
  - G*d and G^T*w from the set over every ray, K times each (device time, mean);
  - ray_project / ray_backproject over the same rays, S sources per call as in tomo_bench (device time, summed);
  - a bit-equality check of the set's results against ray_project / ray_backproject on the first chunk of sources;
  - the wall time of scipy's lsqr over the set's LinearOperator for exactly N iterations (atol = btol = 0), host
    conversions and PCIe copies included.
Prints one JSON line with the card (name, SM clock, power limit from nvidia-smi in the same process).  Every operator
runs once on a small set first (warm-up).  Nothing is written except --out.
"""
import argparse
import json
import pathlib
import subprocess
import sys
import time

import numpy as np

ROOT = pathlib.Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

import uoparallel_seismic_project_b200 as P  # noqa: E402
from uoparallel_seismic_project_b200 import api, workloads as W  # noqa: E402

DIMS = (241, 241, 51)
STARTS = {"config3": 111, "config2": 4}


def card():
    q = "name,clocks.sm,clocks.max.sm,power.limit,power.draw,driver_version"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True, check=True).stdout.strip()
    return dict(zip(q.split(","), [s.strip() for s in out.split(",")]))


def bits_equal(a, b):
    return bool(np.array_equal(np.asarray(a, np.float32).view(np.uint32), np.asarray(b, np.float32).view(np.uint32)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="config3", choices=sorted(STARTS))
    ap.add_argument("--chunk", type=int, default=4, help="sources per ray_project / ray_backproject call")
    ap.add_argument("--reps", type=int, default=5, help="applications of each stored operator")
    ap.add_argument("--lsqr-iters", type=int, default=20)
    ap.add_argument("--out", help="also append the JSON line to this file")
    args = ap.parse_args()
    if P.device_count() < 1:
        sys.exit("rayset_bench: no CUDA device (the ray sets have no CPU fallback)")
    from scipy.sparse.linalg import lsqr
    v = W.heterogeneous_field(DIMS, seed=7)
    v_obs = (v * np.random.default_rng(8).uniform(0.98, 1.02, v.shape)).astype(np.float32)
    pert = np.random.default_rng(9).standard_normal(DIMS).astype(np.float32)
    starts = W.starts(STARTS[args.workload])
    face = np.array([(x, y, 0) for x in range(DIMS[0]) for y in range(DIMS[1])], np.int32)
    chunks = [(s0, min(args.chunk, len(starts) - s0)) for s0 in range(0, len(starts), args.chunk)]
    with P.SweepContext(kernel=api.KERNEL_TILED) as obs_ctx:
        obs_ctx.set_model(v_obs); obs_ctx.set_star(W.star("818")); obs_ctx.set_sources(starts)
        obs_ctx.run()
        observed = np.concatenate([obs_ctx.trace_rays(face, sources=c, max_nodes=1).tt for c in chunks])
    with P.SweepContext(kernel=api.KERNEL_TILED) as ctx:
        ctx.set_model(v); ctx.set_star(W.star("818")); ctx.set_sources(starts)
        ctx.run()
        with ctx.freeze_rays(face[:256], sources=(0, 1)) as warm:   # warm-up of every kernel
            warm.project(pert); warm.backproject(np.ones(warm.shape, np.float32))
        ctx.ray_project(pert, face[:256], sources=(0, 1))
        ctx.ray_backproject(np.ones((1, 256), np.float32), face[:256], sources=(0, 1))

        w0 = time.perf_counter()
        rs = ctx.freeze_rays(face)
        freeze_wall = time.perf_counter() - w0
        residual = np.where(rs.status == api.RAY_OK, observed - rs.tt, 0).astype(np.float32)
        proj_ms, back_ms, exps = [], [], set()
        for _ in range(args.reps):
            proj_ms.append(rs.project(pert).stats.solve_ms)
            bp = rs.backproject(residual)
            back_ms.append(bp.stats.solve_ms)
            exps.add(bp.quantum_exp)

        op_ms = {"project": 0.0, "backproject": 0.0}
        for s0, n in chunks:
            op_ms["project"] += ctx.ray_project(pert, face, sources=(s0, n)).stats.solve_ms
            op_ms["backproject"] += ctx.ray_backproject(residual[s0:s0 + n], face, sources=(s0, n)).stats.solve_ms

        s0, n = chunks[0]
        with ctx.freeze_rays(face, sources=(s0, n)) as part:
            equal = {
                "project": bits_equal(part.project(pert).values, ctx.ray_project(pert, face, sources=(s0, n)).values),
                "backproject": bits_equal(part.backproject(residual[s0:s0 + n]).grad,
                                          ctx.ray_backproject(residual[s0:s0 + n], face, sources=(s0, n)).grad),
            }

        op = rs.as_linear_operator()
        b = residual[rs.status == api.RAY_OK].astype(np.float64)
        w0 = time.perf_counter()
        out = lsqr(op, b, damp=1.0, atol=0.0, btol=0.0, iter_lim=args.lsqr_iters)
        lsqr_wall = time.perf_counter() - w0
        nbytes, entries = rs.nbytes, int(np.where(rs.status == api.RAY_OK, rs.length - 1, 0).sum())
        status = np.bincount(rs.status.ravel(), minlength=6)
        freeze = rs.stats
        rs.close()
    rays = len(starts) * len(face)
    line = {
        "tool": "rayset_bench", "workload": args.workload, "dims": DIMS, "star": "818", "sources": len(starts),
        "receivers_per_source": len(face), "rays": rays,
        "freeze_ms": round(freeze.solve_ms, 3), "freeze_wall_s": round(freeze_wall, 3),
        "freeze_launches": freeze.kernel_launches, "freeze_candidate_evals": freeze.relaxations,
        "nbytes": nbytes, "entries": entries, "mean_edges_per_ray": round(entries / rays, 2),
        "rayset_project_ms": round(float(np.mean(proj_ms)), 3), "rayset_backproject_ms": round(float(np.mean(back_ms)), 3),
        "rayset_project_ms_all": [round(x, 3) for x in proj_ms],
        "rayset_backproject_ms_all": [round(x, 3) for x in back_ms],
        "ray_project_ms": round(op_ms["project"], 3), "ray_backproject_ms": round(op_ms["backproject"], 3),
        "operator_chunk_sources": args.chunk,
        "bit_equal_on_chunk": dict(equal, sources=[s0, n]),
        "quantum_exp": sorted(exps),
        "lsqr_iterations": int(out[2]), "lsqr_wall_s": round(lsqr_wall, 3), "lsqr_damp": 1.0,
        "lsqr_r1norm": float(out[3]), "rhs_norm": float(np.linalg.norm(b)),
        "status_counts": dict(zip(["ok", "unreached", "not_fixed_point", "no_predecessor", "stalled", "truncated"],
                                  status.tolist())),
        "card": card(),
    }
    text = json.dumps(line)
    print(text)
    if args.out:
        with open(args.out, "a") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
