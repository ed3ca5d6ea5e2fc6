#!/usr/bin/env python3
"""refine_bench.py -- sub-node refinement of located events (SweepContext.refine_events / refine_regions) on config 3,
on one GPU.

  python tools/refine_bench.py [--events 1,100,1000,10000] [--subdivs 2,4,8,16,32] [--reps 2]
                               [--accuracy-events 1000] [--no-accuracy] [--out FILE]

Cost.  Config 3 and its events as in tools/locate_bench.py (the 241x241x51 heterogeneous box, seed 7, 818-FS, the 111
start-111 points as stations; picks = the stations' times at a uniform node + U(0, 20) + N(0, 0.05), about 10 % NaN).
For each event count E and subdiv f: the device time of locate_events, of refine_events around the located nodes, and
of refine_regions there at the 95 % levels of sigma = 0.05 (each from the call's stats, mean of --reps calls, one call
from 10,000 events on), beside the float64 bound from the shapes: per lattice point and pick, two evaluations of the
interpolated time (7 lerps of 3 operations) and the formula's 6 operations, at 18.5 T float64 operations per second
(half the B200 data sheet's 37 TFLOPS, which counts a fused multiply-add as two; locate_bench's figure).

Accuracy, against an independent truth.  The config-3 model upsampled 2x (fine[x] = coarse[x div 2] on each axis,
dims 2n - 1, the star at delta / 2), solved for the 111 stations at their doubled positions.  Events at random fine
nodes with at least one odd coordinate (off the coarse nodes); picks = the fine fields there (trace_rays(max_nodes=1),
no field leaves the device) + an origin U(0, 20) + N(0, sigma), sigma in {0, 0.05}.  On the coarse fields: the
median and 90th-percentile position error, in coarse-node units, of locate_events and of the refinement loop of
refine_locations (refine_located) at f = 2, 4, 8; for sigma = 0.05 also the lattice points of the 95 % regions
(refine_regions) against the nodes of misfit_regions.

Prints one JSON line per case with the card (name, SM clock, power limit from nvidia-smi in the same process).  Every
call runs once first (warm-up).  Nothing is written except --out.
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
from locate_bench import DIMS, FP64_OPS, card, make_picks  # noqa: E402

OPS_PER_POINT_PICK = 2 * 7 * 3 + 6


def cube_points(centres, f):
    """Lattice points of each clipped cube."""
    n = 0
    for c in centres:
        ext = 1
        for a in range(3):
            lo = 0 if c[a] > 0 else f
            hi = 2 * f if c[a] < DIMS[a] - 1 else f
            ext *= hi - lo + 1
        n += ext
    return n


def cost(ctx, args, info):
    lines = []
    for nev in (int(x) for x in args.events.split(",")):
        picks = make_picks(ctx, nev, nev)
        reps = 1 if nev >= 10000 else args.reps
        locs = [ctx.locate_events(picks) for _ in range(reps)]
        loc = locs[0]
        loc_ms = float(np.mean([x.stats.solve_ms for x in locs]))
        ok = loc.status == api.LOC_OK
        centres = np.where(ok[:, None], loc.node, 0).astype(np.int32)
        k = (~np.isnan(picks)).sum(1)
        for f in (int(x) for x in args.subdivs.split(",")):
            refs = [ctx.refine_events(picks, centres, f) for _ in range(reps)]
            ref = refs[0]
            levels = P.uncertainty_levels(ref, 0.05)
            regs = [ctx.refine_regions(picks, centres, f, levels) for _ in range(reps)]
            same = all((r.point == ref.point).all() and (r.misfit.view(np.uint32) == ref.misfit.view(np.uint32)).all()
                       for r in refs) and all((r.count == regs[0].count).all() for r in regs)
            ref_ms = float(np.mean([x.stats.solve_ms for x in refs]))
            reg_ms = float(np.mean([x.stats.solve_ms for x in regs]))
            pts = sum(cube_points(centres[e:e + 1], f) * int(k[e]) for e in range(nev) if k[e])
            ops = OPS_PER_POINT_PICK * pts
            line = {
                "tool": "refine_bench", "case": "cost", "workload": "config3", "dims": DIMS, "star": "818",
                "stations": 111, "events": nev, "subdiv": f, "picks": int(k.sum()),
                "locate_ms": round(loc_ms, 3), "refine_ms": round(ref_ms, 3), "regions_ms": round(reg_ms, 3),
                "refine_ms_all": [round(x.stats.solve_ms, 3) for x in refs],
                "refine_over_locate": round(ref_ms / loc_ms, 4),
                "refine_launches": ref.stats.kernel_launches, "repeat_bit_equal": bool(same),
                "point_picks": int(pts), "fp64_ops": int(ops), "fp64_bound_ms": round(ops / FP64_OPS * 1e3, 3),
                "fp64_ops_per_s": round(ops / (ref_ms / 1e3), 1),
                "refined_not_above_located": bool((ref.misfit[ok] <= loc.misfit[ok]).all()),
                "region_points_median": int(np.median(regs[0].count[ok])) if ok.any() else 0,
                "card": info,
            }
            print(json.dumps(line), flush=True)
            lines.append(line)
    return lines


def accuracy(coarse_ctx, v, args, info):
    fine_dims = tuple(2 * n - 1 for n in DIMS)
    fine = v[np.ix_(*[np.arange(m) // 2 for m in fine_dims])]
    stations = W.starts(111)
    lines = []
    with P.SweepContext(kernel=api.KERNEL_TILED) as fctx:
        fctx.set_model(fine); fctx.set_star(W.star("818"), 5.0); fctx.set_sources(2 * np.asarray(stations))
        t = time.perf_counter()
        fctx.run()
        fine_solve_s = time.perf_counter() - t
        rng = np.random.default_rng(2024)
        E = args.accuracy_events
        nodes = np.zeros((0, 3), np.int64)
        while len(nodes) < E:
            cand = np.stack([rng.integers(0, m, 4 * E) for m in fine_dims], 1)
            nodes = np.concatenate([nodes, cand[(cand % 2 == 1).any(1)]])[:E]
        tt = fctx.trace_rays(nodes.astype(np.int32), max_nodes=1).tt.T      # [E, S]
    truth = nodes / 2.0                                                     # coarse-node units
    for sigma in (0.0, 0.05):
        picks = (tt + rng.uniform(0, 20, (E, 1)) + (rng.normal(0, sigma, tt.shape) if sigma else 0)).astype(np.float32)
        loc = coarse_ctx.locate_events(picks)
        ok = loc.status == api.LOC_OK
        err = np.linalg.norm(loc.node - truth, axis=1)[ok]
        line = {"tool": "refine_bench", "case": "accuracy", "workload": "config3 vs 2x upsampled", "fine_dims": fine_dims,
                "fine_solve_s": round(fine_solve_s, 2), "events": E, "sigma": sigma, "located_ok": int(ok.sum()),
                "locate": {"median": round(float(np.median(err)), 4), "p90": round(float(np.percentile(err, 90)), 4)},
                "card": info}
        if sigma:
            reg = coarse_ctx.misfit_regions(picks, P.uncertainty_levels(loc, sigma))
            line["locate"]["region_nodes_median"] = float(np.median(reg.count[ok]))
            line["locate"]["region_nodes_max"] = int(reg.count[ok].max())
        for f in (2, 4, 8):
            ref = P.refine_located(coarse_ctx, picks, loc, subdiv=f)
            okr = ref.status == api.LOC_OK
            e = np.linalg.norm(ref.position - truth, axis=1)[okr]
            r = {"median": round(float(np.median(e)), 4), "p90": round(float(np.percentile(e, 90)), 4),
                 "moves_max": int(ref.moves.max()), "still_on_edge": int(ref.on_edge.sum())}
            if sigma:
                reg = coarse_ctx.refine_regions(picks, ref.centre, f, P.uncertainty_levels(ref, sigma))
                r["region_points_median"] = float(np.median(reg.count[okr]))
                r["region_points_max"] = int(reg.count[okr].max())
                r["region_truncated"] = int(reg.truncated.sum())
                r["region_node_units3_median"] = float(np.median(reg.count[okr])) / f ** 3
            line[f"refine_f{f}"] = r
        print(json.dumps(line), flush=True)
        lines.append(line)
    return lines


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--events", default="1,100,1000,10000")
    ap.add_argument("--subdivs", default="2,4,8,16,32")
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--accuracy-events", type=int, default=1000)
    ap.add_argument("--no-accuracy", action="store_true")
    ap.add_argument("--out", help="also append the JSON lines to this file")
    args = ap.parse_args()
    if P.device_count() < 1:
        sys.exit("refine_bench: no CUDA device (refinement has no CPU fallback)")
    v = W.heterogeneous_field(DIMS, seed=7)
    info = card()
    with P.SweepContext(kernel=api.KERNEL_TILED) as ctx:
        ctx.set_model(v); ctx.set_star(W.star("818")); ctx.set_sources(W.starts(111))
        ctx.run()
        warm = make_picks(ctx, 2, 0)
        wl = ctx.locate_events(warm)
        wc = np.where((wl.status == api.LOC_OK)[:, None], wl.node, 0).astype(np.int32)
        ctx.refine_events(warm, wc, 2); ctx.refine_regions(warm, wc, 2, np.zeros(2, np.float32))
        lines = cost(ctx, args, info)
        if not args.no_accuracy:
            lines += accuracy(ctx, v, args, info)
    if args.out:
        with open(args.out, "a") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
