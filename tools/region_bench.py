#!/usr/bin/env python3
"""region_bench.py -- the misfit regions of located events (SweepContext.misfit_regions) on config 3, on one GPU.

  python tools/region_bench.py [--events 1,100,1000] [--host-max 100] [--sigmas 0.05,1,4] [--reps 3] [--out FILE]

Config 3 and its events as in tools/locate_bench.py: the 241x241x51 heterogeneous box (seed 7), 818-FS, the 111
start-111 points as stations, solved device-resident; per event count E, seeded events (default_rng(E)) with picks =
the stations' times at a uniform node + U(0, 20) + N(0, 0.05), about 10 % NaN.  The levels are those of
location_uncertainty (uncertainty_levels: best misfit + sigma^2 chi2.ppf(0.95, 3)), for each sigma of --sigmas: the
picks' own noise (0.05) gives regions of a node or two, larger sigmas regions of thousands of nodes, whose atomics are
what the kernel adds to the location pass.  In one process it measures:
  - locate_events and misfit_regions: device time from each call's stats (mean of --reps calls);
  - the host route for up to --host-max events: misfit_box per event to the host, then numpy box <= level, the count,
    the 9 integer moments and the bounding box; wall time, and a check that they equal the kernel's.
Prints one JSON line per event count with the card (name, SM clock, power limit from nvidia-smi in the same process).
Every call runs once first (warm-up).  Nothing is written except --out.
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
from locate_bench import DIMS, card, make_picks  # noqa: E402


def host_route(ctx, picks, levels):
    """count [E], moments [E, 9], lo / hi [E, 3] from the misfit box of each event on the host."""
    E = len(picks)
    count = np.zeros(E, np.int64)
    moments = np.zeros((E, 9), np.int64)
    lo = np.full((E, 3), -1, np.int32)
    hi = np.full((E, 3), -1, np.int32)
    for e in range(E):
        if np.isnan(levels[e]):
            continue
        c = np.argwhere(ctx.misfit_box(picks[e]) <= levels[e]).astype(np.int64)
        count[e] = len(c)
        if len(c):
            lo[e], hi[e] = c.min(0), c.max(0)
            moments[e] = [*c.sum(0), *(c * c).sum(0), (c[:, 0] * c[:, 1]).sum(), (c[:, 0] * c[:, 2]).sum(),
                          (c[:, 1] * c[:, 2]).sum()]
    return count, moments, lo, hi


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--events", default="1,100,1000")
    ap.add_argument("--host-max", type=int, default=100, help="largest event count also run by the host route")
    ap.add_argument("--sigmas", default="0.05,1,4")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", help="also append the JSON lines to this file")
    args = ap.parse_args()
    if P.device_count() < 1:
        sys.exit("region_bench: no CUDA device (misfit regions have no CPU fallback)")
    v = W.heterogeneous_field(DIMS, seed=7)
    stations = W.starts(111)
    S = len(stations)
    info = card()
    with P.SweepContext(kernel=api.KERNEL_TILED) as ctx:
        ctx.set_model(v); ctx.set_star(W.star("818")); ctx.set_sources(stations)
        ctx.run()
        warm = make_picks(ctx, 2, 0)
        wl = ctx.locate_events(warm)
        ctx.misfit_regions(warm, P.uncertainty_levels(wl, 1.0)); ctx.misfit_box(warm[0])
        lines = []
        cases = [(int(n), float(sg)) for n in args.events.split(",") for sg in args.sigmas.split(",")]
        for nev, sigma in cases:
            picks = make_picks(ctx, nev, nev)
            locs = [ctx.locate_events(picks) for _ in range(args.reps)]
            levels = P.uncertainty_levels(locs[0], sigma)
            regs = [ctx.misfit_regions(picks, levels) for _ in range(args.reps)]
            reg = regs[0]
            same = all((r.count == reg.count).all() and (r.moments == reg.moments).all() for r in regs)
            loc_ms = float(np.mean([x.stats.solve_ms for x in locs]))
            reg_ms = float(np.mean([x.stats.solve_ms for x in regs]))
            ok = reg.count > 0
            line = {
                "tool": "region_bench", "workload": "config3", "dims": DIMS, "star": "818", "stations": S,
                "events": nev, "sigma": sigma, "confidence": 0.95,
                "locate_ms": round(loc_ms, 3), "regions_ms": round(reg_ms, 3),
                "regions_ms_all": [round(x.stats.solve_ms, 3) for x in regs],
                "regions_over_locate": round(reg_ms / loc_ms, 3),
                "regions_launches": reg.stats.kernel_launches, "regions_d2h_bytes": reg.stats.d2h_bytes,
                "repeat_bit_equal": bool(same),
                "region_nodes_median": int(np.median(reg.count[ok])) if ok.any() else 0,
                "region_nodes_max": int(reg.count.max()) if nev else 0,
                "region_nodes_total": int(reg.count.sum()),
                "status_counts": np.bincount(reg.status, minlength=3).tolist(),
                "card": info,
            }
            if nev <= args.host_max:
                t = time.perf_counter()
                count, moments, lo, hi = host_route(ctx, picks, levels)
                host_s = time.perf_counter() - t
                line["host_route_s"] = round(host_s, 3)
                line["host_route_d2h_bytes"] = int(nev * np.prod(DIMS) * 4)
                line["host_over_regions"] = round(host_s * 1e3 / reg_ms, 1)
                line["host_route_equal"] = bool((count == reg.count).all() and (moments == reg.moments).all()
                                                and (lo == reg.lo).all() and (hi == reg.hi).all())
            else:
                line["host_route_s"] = "not measured"
            print(json.dumps(line), flush=True)
            lines.append(line)
    if args.out:
        with open(args.out, "a") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
