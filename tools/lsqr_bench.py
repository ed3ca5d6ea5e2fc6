#!/usr/bin/env python3
"""lsqr_bench.py -- the LSQR step of a ray set solved on the device (RaySet.lsqr) against scipy's lsqr over the set's
LinearOperator, on one GPU.

  python tools/lsqr_bench.py [--workload config3|config2] [--iters N] [--smooth MU] [--out FILE]

The workloads and residuals of tools/rayset_bench.py: the 241x241x51 heterogeneous box (seed 7), 818-FS, config 3 =
111 starts, config 2 = 4, every receiver of the face z = 0 frozen into one set; "observed" times from a second context
on the model perturbed by U(0.98, 1.02) (seed 8); b = float32(observed - t) over every OK ray.  In one process it
measures, for exactly N iterations (atol = btol = 0, damp = 1):
  - RaySet.lsqr with smooth = 0 and with smooth = MU: device time from the call's stats, and the host wall clock;
  - scipy's lsqr over RaySet.as_linear_operator: the host wall clock (conversions and PCIe copies included);
  - the relative difference of the two x at smooth = 0, and whether istop / itn agree.
Every path runs once for 2 iterations first (warm-up).  Prints one JSON line with the card (name, SM clock, power limit
from nvidia-smi in the same process).  Nothing is written except --out.
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="config3", choices=sorted(STARTS))
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--smooth", type=float, default=1.0)
    ap.add_argument("--out", help="also append the JSON line to this file")
    args = ap.parse_args()
    if P.device_count() < 1:
        sys.exit("lsqr_bench: no CUDA device (the ray sets have no CPU fallback)")
    from scipy.sparse.linalg import lsqr
    v = W.heterogeneous_field(DIMS, seed=7)
    v_obs = (v * np.random.default_rng(8).uniform(0.98, 1.02, v.shape)).astype(np.float32)
    starts = W.starts(STARTS[args.workload])
    face = np.array([(x, y, 0) for x in range(DIMS[0]) for y in range(DIMS[1])], np.int32)
    chunks = [(s0, min(4, len(starts) - s0)) for s0 in range(0, len(starts), 4)]
    with P.SweepContext(kernel=api.KERNEL_TILED) as obs_ctx:
        obs_ctx.set_model(v_obs); obs_ctx.set_star(W.star("818")); obs_ctx.set_sources(starts)
        obs_ctx.run()
        observed = np.concatenate([obs_ctx.trace_rays(face, sources=c, max_nodes=1).tt for c in chunks])
    with P.SweepContext(kernel=api.KERNEL_TILED) as ctx:
        ctx.set_model(v); ctx.set_star(W.star("818")); ctx.set_sources(starts)
        ctx.run()
        rs = ctx.freeze_rays(face)
        rows = rs.status == api.RAY_OK
        b = (observed - rs.tt).astype(np.float32)[rows].astype(np.float64)
        op = rs.as_linear_operator(rows)
        kw = dict(damp=1.0, atol=0.0, btol=0.0)
        rs.lsqr(b, rows, smooth=args.smooth, iter_lim=2, **kw)    # warm-up
        lsqr(op, b, iter_lim=2, **kw)
        dev = {}
        for mu in (0.0, args.smooth):
            w0 = time.perf_counter()
            sol = rs.lsqr(b, rows, smooth=mu, iter_lim=args.iters, **kw)
            wall = time.perf_counter() - w0
            dev[mu] = (sol, wall)
        w0 = time.perf_counter()
        ref = lsqr(op, b, iter_lim=args.iters, **kw)
        scipy_wall = time.perf_counter() - w0
        nrays, nbytes = rs.status.size, rs.nbytes
        rs.close()
    m, D = int(rows.sum()), int(np.prod(DIMS))
    nx, ny, nz = DIMS
    mD = (nx - 1) * ny * nz + nx * (ny - 1) * nz + nx * ny * (nz - 1)
    x0 = dev[0.0][0].x.ravel()

    def entry(mu):
        sol, wall = dev[mu]
        rows_u = m + (mD if mu > 0 else 0)
        return {"smooth": mu, "device_ms": round(sol.stats.solve_ms, 3), "wall_s": round(wall, 4),
                "ms_per_iteration": round(sol.stats.solve_ms / max(sol.itn, 1), 3), "itn": sol.itn, "istop": sol.istop,
                "r1norm": sol.r1norm, "launches": sol.stats.kernel_launches, "d2h_bytes": sol.stats.d2h_bytes,
                "h2d_bytes": sol.stats.h2d_bytes, "u_rows": rows_u,
                "workspace_bytes": 8 * rows_u + 24 * D + 8 * m + 8 * ((max(rows_u, D) + 2047) // 2048 + 1)}

    line = {
        "tool": "lsqr_bench", "workload": args.workload, "dims": DIMS, "star": "818", "sources": len(starts),
        "rays": nrays, "rows": m, "rayset_nbytes": nbytes, "iterations": args.iters, "damp": 1.0,
        "device": [entry(0.0), entry(args.smooth)],
        "scipy_wall_s": round(scipy_wall, 4), "scipy_itn": int(ref[2]), "scipy_istop": int(ref[1]),
        "scipy_r1norm": float(ref[3]),
        "x_rel_diff_vs_scipy": float(np.linalg.norm(x0 - ref[0]) / np.linalg.norm(ref[0])),
        "speedup_wall": round(scipy_wall / dev[0.0][1], 2),
        "card": card(),
    }
    text = json.dumps(line)
    print(text)
    if args.out:
        with open(args.out, "a") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
