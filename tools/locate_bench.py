#!/usr/bin/env python3
"""locate_bench.py -- event location by grid search over config 3's 111 station fields, on one GPU.

  python tools/locate_bench.py [--events 1,100,1000,10000] [--torch-max 1000] [--reps 3] [--out FILE]

Config 3: the 241x241x51 heterogeneous box (seed 7), 818-FS, the 111 start-111 points as stations, solved
device-resident.  For each event count E, seeded events (numpy default_rng(E)): a node drawn uniformly, an origin time
U(0, 20), picks = the stations' times there (read with trace_rays(max_nodes=1), no field leaves the device) plus
N(0, 0.05) noise, and about 10 % of the picks NaN.  In one process it measures:
  - locate_events: device time from the call's stats (mean of --reps calls, one for 10,000 events) and events/s;
  - what the kernel needs, from the shapes: HBM bytes (every station's field read once per launch) and float64
    operations (6 per pick and node: two passes; the division and the argmin are left out), and which bound is larger
    on a B200 (7.7 TB/s; 18.5 T float64 additions or multiplications per second, half the data sheet's 37 TFLOPS,
    which counts a fused multiply-add as two);
  - the same misfits from a plain torch float64 implementation on the same device (fields as one [S, D] float32
    tensor, per event r = obs - tt over the picked stations, t0 = sum / k, misfit = sum of (r - t0)^2), timed with CUDA
    events for up to --torch-max events, and the largest difference between its per-event minimum and the kernel's.
Prints one JSON line per event count with the card (name, SM clock, power limit from nvidia-smi in the same process).
Every kernel runs once first (warm-up).  Nothing is written except --out.
"""
import argparse
import json
import pathlib
import subprocess
import sys

import numpy as np

ROOT = pathlib.Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

import uoparallel_seismic_project_b200 as P  # noqa: E402
from uoparallel_seismic_project_b200 import api, workloads as W  # noqa: E402

DIMS = (241, 241, 51)
HBM_BPS = 7.7e12
FP64_OPS = 18.5e12


def card():
    q = "name,clocks.sm,clocks.max.sm,power.limit,power.draw,driver_version"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True, check=True).stdout.strip()
    return dict(zip(q.split(","), [s.strip() for s in out.split(",")]))


def make_picks(ctx, nev, seed):
    rng = np.random.default_rng(seed)
    nodes = np.stack(np.unravel_index(rng.integers(int(np.prod(DIMS)), size=nev), DIMS), 1).astype(np.int32)
    tt = ctx.trace_rays(nodes, max_nodes=1).tt.T          # [E, S]: the times at the event nodes, whatever the status
    picks = (tt + rng.uniform(0, 20, (nev, 1)) + rng.normal(0, 0.05, tt.shape)).astype(np.float32)
    picks[rng.random(picks.shape) < 0.1] = np.nan
    return picks


def torch_misfits(fields, picks):
    """Per-event minimum misfit and the device time of a plain torch float64 implementation."""
    import torch
    mins = np.empty(len(picks), np.float32)
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    p_all = torch.from_numpy(picks).cuda()
    start.record()
    out = []
    for e in range(len(picks)):
        idx = torch.nonzero(~torch.isnan(p_all[e])).squeeze(1)
        tt = fields.index_select(0, idx).double()
        r = p_all[e, idx].double().unsqueeze(1) - tt
        t0 = r.sum(0) / idx.numel()
        m = ((r - t0) ** 2).sum(0).float()
        m[torch.isinf(tt).any(0)] = float("inf")
        out.append(m.min())
    res = torch.stack(out)
    stop.record()
    torch.cuda.synchronize()
    mins[:] = res.cpu().numpy()
    return mins, start.elapsed_time(stop)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--events", default="1,100,1000,10000")
    ap.add_argument("--torch-max", type=int, default=1000, help="largest event count also run by the torch baseline")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", help="also append the JSON lines to this file")
    args = ap.parse_args()
    if P.device_count() < 1:
        sys.exit("locate_bench: no CUDA device (event location has no CPU fallback)")
    import torch
    v = W.heterogeneous_field(DIMS, seed=7)
    stations = W.starts(111)
    S, D = len(stations), int(np.prod(DIMS))
    info = card()
    with P.SweepContext(kernel=api.KERNEL_TILED) as ctx:
        ctx.set_model(v); ctx.set_star(W.star("818")); ctx.set_sources(stations)
        ctx.run()
        fields = torch.from_numpy(np.stack([ctx.get_tt(s) for s in range(S)]).reshape(S, D)).cuda()
        warm = make_picks(ctx, 2, 0)
        ctx.locate_events(warm); ctx.misfit_box(warm[0]); torch_misfits(fields, warm)
        lines = []
        for nev in (int(x) for x in args.events.split(",")):
            picks = make_picks(ctx, nev, nev)
            reps = 1 if nev >= 10000 else args.reps
            runs = [ctx.locate_events(picks) for _ in range(reps)]
            loc = runs[0]
            ms = [r.stats.solve_ms for r in runs]
            same = all((r.node == loc.node).all() and (r.misfit.view(np.uint32) == loc.misfit.view(np.uint32)).all()
                       for r in runs)
            k = int(np.isfinite(picks).sum())
            chunks = loc.stats.kernel_launches - 1
            hbm = chunks * S * D * 4 + k * 12 + nev * 64
            ops = 6 * k * D
            line = {
                "tool": "locate_bench", "workload": "config3", "dims": DIMS, "star": "818", "stations": S,
                "events": nev, "picks": k, "launches": loc.stats.kernel_launches,
                "device_ms": round(float(np.mean(ms)), 3), "device_ms_all": [round(x, 3) for x in ms],
                "events_per_s": round(nev / (np.mean(ms) / 1e3), 1), "repeat_bit_equal": bool(same),
                "hbm_bytes": hbm, "fp64_ops": ops,
                "hbm_bound_ms": round(hbm / HBM_BPS * 1e3, 3), "fp64_bound_ms": round(ops / FP64_OPS * 1e3, 3),
                "bound": "fp64" if ops / FP64_OPS > hbm / HBM_BPS else "hbm",
                "fp64_ops_per_s": round(ops / (np.mean(ms) / 1e3), 1),
                "status_counts": np.bincount(loc.status, minlength=3).tolist(),
                "card": info,
            }
            if nev <= args.torch_max:
                mins, tms = torch_misfits(fields, picks)
                ok = loc.status == api.LOC_OK
                line["torch_ms"] = round(tms, 3)
                line["torch_over_kernel"] = round(tms / np.mean(ms), 2)
                line["torch_max_abs_diff"] = float(np.max(np.abs(mins[ok].astype(np.float64) - loc.misfit[ok])))
                line["torch_max_rel_diff"] = float(np.max(np.abs(mins[ok].astype(np.float64) - loc.misfit[ok])
                                                          / np.maximum(loc.misfit[ok], 1e-30)))
            else:
                line["torch_ms"] = "not measured"
            print(json.dumps(line), flush=True)
            lines.append(line)
    if args.out:
        with open(args.out, "a") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
