#!/usr/bin/env python3
"""tomo_bench.py -- the tomography operators over the rays from every node of the z = 0 face, on one GPU.

  python tools/tomo_bench.py [--workload config3|config2] [--chunk S] [--out FILE]

Solves the workload device-resident (241x241x51 heterogeneous box, seed 7, 818-FS; config 3 = start-111, config 2 =
start-4), and a second context solves the same starts in a perturbed model (slowness x U(0.98, 1.02), seed 8) for
"observed" receiver times.  Then, S sources per call (default 4), over the 241 x 241 = 58,081 receivers of the face
z = 0: trace_rays with max_nodes = 1 (the receiver table that misfit_gradient reads), ray_project of a random
perturbation and ray_backproject of the residuals (predicted - observed).  Prints one JSON line: device times (CUDA
events, the calls' own stats) of each operator, rays/s, candidate evaluations, the quantum exponents, the statuses and
the card (name, SM clock, power limit from nvidia-smi in the same process).  Every operator runs once on a small
receiver set first (warm-up).  Nothing is written except --out.
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
    ap.add_argument("--chunk", type=int, default=4, help="sources per operator call")
    ap.add_argument("--out", help="also append the JSON line to this file")
    args = ap.parse_args()
    if P.device_count() < 1:
        sys.exit("tomo_bench: no CUDA device (the operators have no CPU fallback)")
    v = W.heterogeneous_field(DIMS, seed=7)
    v_obs = (v * np.random.default_rng(8).uniform(0.98, 1.02, v.shape)).astype(np.float32)
    pert = np.random.default_rng(9).standard_normal(DIMS).astype(np.float32)
    starts = W.starts(STARTS[args.workload])
    face = np.array([(x, y, 0) for x in range(DIMS[0]) for y in range(DIMS[1])], np.int32)
    chunks = [(s0, min(args.chunk, len(starts) - s0)) for s0 in range(0, len(starts), args.chunk)]
    with P.SweepContext(kernel=api.KERNEL_TILED) as obs_ctx:
        obs_ctx.set_model(v_obs); obs_ctx.set_star(W.star("818")); obs_ctx.set_sources(starts)
        obs_ctx.run()
        observed = [obs_ctx.trace_rays(face, sources=c, max_nodes=1).tt for c in chunks]
    t = {"table": 0.0, "project": 0.0, "backproject": 0.0}
    evals = {k: 0 for k in t}
    wall = dict(t)
    exps, status = [], np.zeros(6, np.int64)
    with P.SweepContext(kernel=api.KERNEL_TILED) as ctx:
        ctx.set_model(v); ctx.set_star(W.star("818")); ctx.set_sources(starts)
        ctx.run()                                   # warm-up solve
        solve = ctx.run()
        ctx.trace_rays(face[:256], sources=(0, 1), max_nodes=1)   # warm-up of every operator
        ctx.ray_project(pert, face[:256], sources=(0, 1))
        ctx.ray_backproject(np.ones((1, 256), np.float32), face[:256], sources=(0, 1))
        for c, obs in zip(chunks, observed):
            w0 = time.perf_counter()
            tab = ctx.trace_rays(face, sources=c, max_nodes=1)
            w1 = time.perf_counter()
            pr = ctx.ray_project(pert, face, sources=c)
            w2 = time.perf_counter()
            res = np.where(np.isfinite(tab.tt - obs), tab.tt - obs, 0).astype(np.float32)
            w3 = time.perf_counter()
            bp = ctx.ray_backproject(res, face, sources=c)
            w4 = time.perf_counter()
            for k, r, dt in (("table", tab, w1 - w0), ("project", pr, w2 - w1), ("backproject", bp, w4 - w3)):
                t[k] += r.stats.solve_ms
                evals[k] += r.stats.relaxations
                wall[k] += dt
            exps.append(bp.quantum_exp)
            status += np.bincount(pr.status.ravel(), minlength=6)
    rays = len(starts) * len(face)
    line = {
        "tool": "tomo_bench", "workload": args.workload, "dims": DIMS, "star": "818", "sources": len(starts),
        "receivers_per_source": len(face), "chunk_sources": args.chunk, "calls_per_operator": len(chunks),
        "rays": rays, "solve_ms": round(solve.solve_ms, 3),
        "receiver_table_ms": round(t["table"], 3), "project_ms": round(t["project"], 3),
        "backproject_ms": round(t["backproject"], 3),
        "project_rays_per_s": round(rays / (t["project"] / 1e3)),
        "backproject_rays_per_s": round(rays / (t["backproject"] / 1e3)),
        "candidate_evals": evals,
        "wall_s": {k: round(x, 3) for k, x in wall.items()},
        "quantum_exp_range": [min(exps), max(exps)],
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
