#!/usr/bin/env python3
"""ray_bench.py -- rays from every node of the z = 0 face back to every source, on one GPU.

  python tools/ray_bench.py [--workload config3|config2] [--chunk S] [--out FILE]

Solves the workload device-resident (241x241x51 heterogeneous box, seed 7, 818-FS; config 3 = start-111, config 2 =
start-4), then traces the 241 x 241 = 58,081 receivers of the face z = 0 for every source through
SweepContext.trace_rays, S sources per call (default max_nodes = nx+ny+nz, so every call also copies the rays' nodes
to the host).  Prints one JSON line: solve and trace device times (CUDA events), rays/s, nodes/s, candidate
evaluations/s, mean and maximum ray length, the statuses, the device->host bytes and time, and the card (name, SM
clock, power limit from nvidia-smi in the same process).  The solve is run once untimed first, and one small trace
warms the tracer up.  Nothing is written except --out.
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
    ap.add_argument("--chunk", type=int, default=4, help="sources per trace call")
    ap.add_argument("--out", help="also append the JSON line to this file")
    args = ap.parse_args()
    if P.device_count() < 1:
        sys.exit("ray_bench: no CUDA device (the tracer has no CPU fallback)")
    v = W.heterogeneous_field(DIMS, seed=7)
    starts = W.starts(STARTS[args.workload])
    face = np.array([(x, y, 0) for x in range(DIMS[0]) for y in range(DIMS[1])], np.int32)
    with P.SweepContext(kernel=api.KERNEL_TILED) as ctx:
        ctx.set_model(v); ctx.set_star(W.star("818")); ctx.set_sources(starts)
        ctx.run()                                   # warm-up solve
        solve = ctx.run()
        ctx.trace_rays(face[:256], sources=(0, 1))  # warm-up trace
        t_ms = d2h_ms = 0.0
        rays = nodes = evals = d2h_bytes = 0
        lmax, status = 0, np.zeros(6, np.int64)
        t0 = time.perf_counter()
        for s0 in range(0, len(starts), args.chunk):
            r = ctx.trace_rays(face, sources=(s0, min(args.chunk, len(starts) - s0)))
            t_ms += r.stats.solve_ms
            d2h_ms += r.stats.d2h_ms
            d2h_bytes += r.stats.d2h_bytes
            evals += r.stats.relaxations
            rays += r.length.size
            nodes += int(r.length.sum())
            lmax = max(lmax, int(r.length.max()))
            status += np.bincount(r.status.ravel(), minlength=6)
        wall = time.perf_counter() - t0
    line = {
        "tool": "ray_bench", "workload": args.workload, "dims": DIMS, "star": "818", "sources": len(starts),
        "receivers_per_source": len(face), "chunk_sources": args.chunk,
        "solve_ms": round(solve.solve_ms, 3),
        "trace_ms": round(t_ms, 3), "trace_calls": -(-len(starts) // args.chunk),
        "rays": rays, "nodes": nodes, "candidate_evals": evals,
        "rays_per_s": round(rays / (t_ms / 1e3)), "nodes_per_s": round(nodes / (t_ms / 1e3)),
        "evals_per_s": round(evals / (t_ms / 1e3)),
        "evals_per_step": round(evals / max(1, nodes - rays), 1),
        "mean_length": round(nodes / rays, 3), "max_length": lmax,
        "status_counts": dict(zip(["ok", "unreached", "not_fixed_point", "no_predecessor", "stalled", "truncated"],
                                  status.tolist())),
        "d2h_bytes": d2h_bytes, "d2h_ms": round(d2h_ms, 3), "wall_s_trace_calls": round(wall, 3),
        "card": card(),
    }
    text = json.dumps(line)
    print(text)
    if args.out:
        with open(args.out, "a") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
