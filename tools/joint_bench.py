#!/usr/bin/env python3
"""joint_bench.py -- one joint slowness + hypocentre LSQR step (RaySet.lsqr with hypo=, sweeptt_rayset_lsqr_hypo)
against the plain slowness-only step on the same ray set, on one GPU.

  python tools/joint_bench.py [--events 1000 10000] [--iters N] [--out FILE]

Workload: config 3's model (241x241x51 heterogeneous, seed 7, 818-FS) with its 111 start points as stations.  True
event nodes and picks follow tools/locate_bench.py's make_picks on the model perturbed by U(0.98, 1.02) (seed 8):
origin U(0, 20), N(0, 0.05) noise, about 10 % NaN.  For every event count, in one process:
  - locate the events on the unperturbed model, freeze the station-to-event rays (time of the freeze) and compute
    hypocentre_partials (its time);
  - the joint step and the plain step on the same set and rows for exactly N iterations (atol = btol = 0, damp = 1):
    device time per iteration from the calls' stats, and the workspace bytes of both from the header's formulas;
  - against the true nodes, the median position error (Euclidean, in nodes) after locating, after applying the joint
    step's shifts rounded to nodes, and after one velocity-only step (the plain step's update added to the slowness,
    re-solved) followed by relocation.
Every path runs once for 2 iterations first (warm-up).  Prints one JSON line per event count with the card (name, SM
clock, power limit from nvidia-smi in the same process).  Nothing is written except --out.
"""
import argparse
import json
import pathlib
import sys
import time

import numpy as np

ROOT = pathlib.Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))

import uoparallel_seismic_project_b200 as P  # noqa: E402
from uoparallel_seismic_project_b200 import api, workloads as W  # noqa: E402
from locate_bench import DIMS, card  # noqa: E402

STATIONS = 111


def make_events(ctx, nev, seed):
    """locate_bench.make_picks, keeping the true nodes."""
    rng = np.random.default_rng(seed)
    nodes = np.stack(np.unravel_index(rng.integers(int(np.prod(DIMS)), size=nev), DIMS), 1).astype(np.int32)
    tt = ctx.trace_rays(nodes, max_nodes=1).tt.T
    picks = (tt + rng.uniform(0, 20, (nev, 1)) + rng.normal(0, 0.05, tt.shape)).astype(np.float32)
    picks[rng.random(picks.shape) < 0.1] = np.nan
    return nodes, picks


def median_error(nodes, true, ok):
    return float(np.median(np.linalg.norm((nodes - true)[ok].astype(np.float64), axis=1)))


def workspace(m, D, mu=0, nrec=0):
    """The header's workspace formulas (sweeptt_rayset_lsqr, and _hypo when nrec > 0)."""
    n = D + 4 * nrec
    base = 8 * (m + mu) + 24 * n + 8 * m + 8 * ((max(m + mu, n) + 2047) // 2048 + 1)
    return base + (32 * m + 8 * m + 8 * (nrec + 1) if nrec else 0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--events", type=int, nargs="+", default=[1000, 10000])
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--out", help="also append the JSON lines to this file")
    args = ap.parse_args()
    if P.device_count() < 1:
        sys.exit("joint_bench: no CUDA device (the ray sets have no CPU fallback)")
    v = W.heterogeneous_field(DIMS, seed=7)
    v_obs = (v * np.random.default_rng(8).uniform(0.98, 1.02, v.shape)).astype(np.float32)
    stations = W.starts(STATIONS)
    star = W.star("818")
    D = int(np.prod(DIMS))
    kw = dict(damp=1.0, atol=0.0, btol=0.0)
    for nev in args.events:
        with P.SweepContext(kernel=api.KERNEL_TILED) as obs_ctx:
            obs_ctx.set_model(v_obs); obs_ctx.set_star(star); obs_ctx.set_sources(stations)
            obs_ctx.run()
            true, picks = make_events(obs_ctx, nev, 8)
        with P.SweepContext(kernel=api.KERNEL_TILED) as ctx:
            ctx.set_model(v); ctx.set_star(star); ctx.set_sources(stations)
            ctx.run()
            loc = ctx.locate_events(picks)
            ok = loc.status == api.LOC_OK
            c = np.where(ok[:, None], loc.node, 0).astype(np.int32)
            w0 = time.perf_counter()
            rs = ctx.freeze_rays(c)
            freeze_s = time.perf_counter() - w0
            w0 = time.perf_counter()
            d = P.hypocentre_partials(ctx, c)
            partials_s = time.perf_counter() - w0
            obs = picks.T.astype(np.float64)
            with np.errstate(invalid="ignore"):
                b = (obs - loc.origin_time) - rs.tt.astype(np.float64)
            rows = np.isfinite(obs) & (rs.status == api.RAY_OK) & ok
            h = np.concatenate([d.transpose(1, 0, 2)[rows], np.ones((int(rows.sum()), 1))], axis=1)
            rs.lsqr(b[rows], rows, hypo=h, iter_lim=2, **kw)      # warm-up
            rs.lsqr(b[rows], rows, iter_lim=2, **kw)
            joint = rs.lsqr(b[rows], rows, hypo=h, iter_lim=args.iters, **kw)
            plain = rs.lsqr(b[rows], rows, iter_lim=args.iters, **kw)
            freeze_stats = rs.stats
            rs.close()
        moved = np.clip(np.rint(c + joint.hypo[:, :3]).astype(np.int64), 0, np.array(DIMS) - 1)
        v_step = np.maximum(v + plain.x.astype(np.float32), np.float32(1e-6)).astype(np.float32)
        with P.SweepContext(kernel=api.KERNEL_TILED) as ctx2:
            ctx2.set_model(v_step); ctx2.set_star(star); ctx2.set_sources(stations)
            ctx2.run()
            reloc = ctx2.locate_events(picks)
        ok2 = ok & (reloc.status == api.LOC_OK)
        m = int(rows.sum())
        line = {
            "tool": "joint_bench", "dims": DIMS, "star": "818", "stations": STATIONS, "events": nev,
            "events_located": int(ok.sum()), "rows": m, "iterations": args.iters, "damp": 1.0,
            "joint": {"device_ms": round(joint.stats.solve_ms, 3), "itn": joint.itn,
                      "ms_per_iteration": round(joint.stats.solve_ms / max(joint.itn, 1), 3),
                      "launches": joint.stats.kernel_launches, "workspace_bytes": workspace(m, D, nrec=nev),
                      "r1norm": joint.r1norm},
            "plain": {"device_ms": round(plain.stats.solve_ms, 3), "itn": plain.itn,
                      "ms_per_iteration": round(plain.stats.solve_ms / max(plain.itn, 1), 3),
                      "launches": plain.stats.kernel_launches, "workspace_bytes": workspace(m, D),
                      "r1norm": plain.r1norm},
            "freeze_wall_s": round(freeze_s, 4), "freeze_device_ms": round(freeze_stats.solve_ms, 3),
            "partials_wall_s": round(partials_s, 4),
            "median_error_nodes": {"located": median_error(loc.node, true, ok),
                                   "joint_step_shifted": median_error(moved, true, ok),
                                   "velocity_step_relocated": median_error(reloc.node, true, ok2)},
            "card": card(),
        }
        text = json.dumps(line)
        print(text, flush=True)
        if args.out:
            with open(args.out, "a") as f:
                f.write(text + "\n")


if __name__ == "__main__":
    main()
