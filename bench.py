#!/usr/bin/env python3
"""bench.py -- the benchmark of the multi-start forward-star sweep.

  python bench.py --gpus N --steps K --warmup W            (N>1: launched by torchrun, one rank per GPU)
  python bench.py --impl reference --gpus N --steps K --warmup W
  python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR   (also save what the last timed step computed)

Workload (BASELINE.json configs[2] -- the configuration the metric "... 241x241x51 818-FS, 1/2/4/8 B200" is quoted
on; it fits one GPU): 241x241x51 heterogeneous slowness box (synthetic stand-in, seed 7: the reference's velocity
files are missing blobs), docs/818-FS.txt, docs/start-111-241-241-51.txt.  One *step* = one complete multi-start
solve of all 111 sources (travel times re-initialised, relaxed to the fixed point).  N>1 is STRONG scaling: the 111
sources are dealt round-robin to the ranks (rank r: sources r, r+N, ...; the mpi/backup.c:351-363 scheme), each rank
solves its share on its own replica of the box -- no data-path collective; the ideal speed-up at 8 GPUs is 111/14.
`--workload config2` is BASELINE configs[1] (start-4; weak scaling: 4 private sources per GPU); at N=1 it also
rides along under "extras" together with config 1 (3-FS) and the 5-FS star.

Prints ONE JSON line (rank 0).  metric = GRelax/s: in-bounds (node, offset, source) pull
evaluations executed per second, summed over GPUs; converged sources/s rides along.

--dump-outputs DIR writes the travel-time fields of the last timed step, sampled at the same seeded node set for every
source (see dump_outputs), as DIR/tt.npy (DIR/tt_rank<r>.npy per rank when N>1).  The inputs are fixed by their seeds,
so two builds run with the same arguments can be compared output for output.  It applies to --impl ours only: the
reference arm times the original serial sweepXYZ over slices of the star and never holds a converged field of this
project to dump.
"""
import argparse
import ctypes
import hashlib
import json
import os
import re
import statistics
import subprocess
import sys
import time
import pathlib

ROOT = pathlib.Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

DIMS = (241, 241, 51)
WORKLOADS = {
    "config3": "241x241x51 heterogeneous slowness (synthetic, seed 7), 818-FS, start-111 (111 sources) sharded over the GPUs",
    "config2": "241x241x51 heterogeneous slowness (synthetic, seed 7), 818-FS, start-4 (4 sources per GPU)",
    "config4": "1201x1201x251 heterogeneous slowness (synthetic, seed 11), 818-FS, 24 sources (start-24 x5) sharded over the GPUs",
}
VISITS_PER_SWEEP_818 = 2_246_171_812   # in-bounds (node, offset) visits of one reference sweep of the 241 box (SURVEY 8a)
DUMP_NODES = 1 << 16   # sampled nodes per source: 111 sources x 64 Ki x 4 B = 29 MB, under the 64 MB a dump may take


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the config-1 / config-2 / 5-FS riders at N=1")
    ap.add_argument("--workload", default="config3", choices=["config2", "config3", "config4"],
                    help="config3 (default, the contract's workload): 241 box, start-111 sharded over the GPUs (strong); "
                         "config2: 241 box, 4 sources per GPU (weak); "
                         "config4: 1201x1201x251, 24 sources sharded over the GPUs (strong, device-resident only). "
                         "Config 5 (one source, one huge grid over all GPUs) is tools/config5_bench.py.")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, save a seeded sample of the travel times of the last timed step as "
                         "float32 .npy files in DIR")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs saves the GPU solve's fields: it needs --impl ours")
    return args


# ------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock, power and throttle reasons DURING the timed region: NVML polled every 2 ms from a thread
    (the timed region of config 2 is ~0.3 s, too short for `nvidia-smi -lms`), nvidia-smi as the fallback."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.p = None
        self.thread = None
        self.rows = []          # (sm MHz, max MHz, watts, reasons bitmask)
        self._stop = False
        try:
            import threading
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.thread = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "50", "-i", str(index)], stdout=subprocess.PIPE,
                                      stderr=subprocess.DEVNULL, text=True)
        except OSError:
            pass

    def _poll(self):
        nv = self.nv
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
            getattr(nv, "nvmlDeviceGetCurrentClocksThrottleReasons", None)
        while not self._stop:
            try:
                sm = float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                pw = nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0
                rs = int(get_reasons(self.h)) if get_reasons else 0
                self.rows.append((sm, self.mx, pw, rs))
            except Exception:
                pass
            time.sleep(0.002)

    def _stop_nvml(self):
        self._stop = True
        self.thread.join(timeout=2)
        nv = self.nv
        def bit(name, default):
            return getattr(nv, "nvmlClocksEventReason" + name, getattr(nv, "nvmlClocksThrottleReason" + name, default))
        bits = {"hw_slowdown": bit("HwSlowdown", 0x8), "hw_thermal_slowdown": bit("HwThermalSlowdown", 0x40),
                "sw_thermal_slowdown": bit("SwThermalSlowdown", 0x20), "sw_power_cap": bit("SwPowerCap", 0x4)}
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm = [r[0] for r in self.rows]; pw = [r[2] for r in self.rows]
        reasons = sorted(n for n, b in bits.items() if any(r[3] & b for r in self.rows))
        load = [c for c, p in zip(sm, pw) if p >= 0.5 * max(pw)] or sm
        return {"sm_mhz": statistics.median(load), "sm_max_mhz": self.mx, "reasons": reasons,
                "samples": len(sm), "power_w_max": max(pw), "source": "nvml, 2 ms period"}

    def stop(self):
        if self.thread is not None:
            return self._stop_nvml()
        if not self.p:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            out = self.p.communicate(timeout=5)[0]
        except subprocess.TimeoutExpired:
            self.p.kill()
            out = self.p.communicate()[0]
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for n, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        load = [c for c, p in zip(sm, pw) if p >= 0.5 * max(pw)] or sm
        return {"sm_mhz": statistics.median(load), "sm_max_mhz": max(mx), "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(pw), "source": "nvidia-smi -lms 50"}


# ------------------------------------------------------------------------------------------
# reference arm / CPU baseline: the reference's own serial code on the host cores
# ------------------------------------------------------------------------------------------
def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def _cpu_worker(args):
    """One process per source (the mpi/backup.c scheme): time consecutive calls of the reference's sweepXYZ over
    1/8 slices of the star (state carried from call to call)."""
    src, slices, kind = args
    import numpy as np
    import oracle
    from uoparallel_seismic_project_b200 import workloads as W
    v = W.heterogeneous_field(DIMS, 7)
    off = np.ascontiguousarray(W.star("818"), np.int32)
    L = len(off) - 1
    nslice = 8
    bounds = [L * i // nslice for i in range(nslice + 1)]
    out = []
    if kind == "reference":
        lib = oracle.reference()
        lib.refh_set_star(ctypes.c_void_p(off.ctypes.data), len(off))
        lib.refh_set_velocity(ctypes.c_void_p(v.ctypes.data), *DIMS)
        lib.refh_init_source(0, int(src[0]), int(src[1]), int(src[2]))
        for k in slices:
            a, b = bounds[k % nslice], bounds[k % nslice + 1]
            t0 = time.perf_counter()
            lib.sweepXYZ(DIMS[0], DIMS[1], DIMS[2], 0, a, b)   # the reference's own function
            out.append((time.perf_counter() - t0, oracle.visits_per_sweep(DIMS, off[a:b], used=b - a)))
    else:
        lib = oracle.restatement()
        d = oracle.star_distances(off)
        tt = oracle.init_tt(DIMS, src)
        for k in slices:
            a, b = bounds[k % nslice], bounds[k % nslice + 1]
            t0 = time.perf_counter()
            lib.oracle_sweep(ctypes.c_void_p(v.ctypes.data), ctypes.c_void_p(tt.ctypes.data), DIMS[0], DIMS[1],
                             DIMS[2], ctypes.c_void_p(off[a:b].ctypes.data), ctypes.c_void_p(d[a:b].ctypes.data),
                             b - a, int(src[0]), int(src[1]), int(src[2]))
            out.append((time.perf_counter() - t0, oracle.visits_per_sweep(DIMS, off[a:b], used=b - a)))
    return out


def cpu_reference_run(steps, warmup, workload):
    """All host cores, one source per process (config 3 has 111 sources to hand out, config 2 has 4).
    Returns (per-step seconds = max over the processes, visits per step, kind, cores)."""
    import multiprocessing as mp
    import oracle
    from uoparallel_seismic_project_b200 import workloads as W
    kind = "reference" if oracle.reference() is not None else "port"
    if kind == "port":
        oracle.restatement()
    starts = W.starts(4) if workload == "config2" else W.starts(111)
    cores = max(1, min(len(starts), host_cores()))
    starts = starts[:cores]
    slices = list(range(warmup + steps))
    ctx = mp.get_context("spawn")
    with ctx.Pool(cores) as pool:
        res = pool.map(_cpu_worker, [(tuple(int(c) for c in s), slices, kind) for s in starts])
    step_s, step_v = [], []
    for k in range(warmup, warmup + steps):
        step_s.append(max(r[k][0] for r in res))
        step_v.append(sum(r[k][1] for r in res))
    return step_s, step_v, kind, cores


def _ref_sweeps_per_source():
    """Sweep counts of the reference's own converged runs on this workload (tests/golden, made by tools/make_golden.py)."""
    n = []
    for name in ("full_241.json", "full_241_more.json", "config3_all.json"):
        try:
            for g in json.loads((ROOT / "tests" / "golden" / name).read_text()):
                if g.get("star") == "818" and g.get("kind") == "hetero" and g.get("seed") == 7 and \
                        tuple(g.get("dims", DIMS)) == DIMS:
                    n.append(g["ref_sweeps"])
        except Exception:
            pass
    return n


def cpu_sample_text(cores, workload):
    return (f"each step = one call of the reference's sweepXYZ per source over 1/8 of the 818-FS offsets (slices rotate, "
            f"state carried across steps), {cores} sources in {cores} processes on {cores} host cores (the mpi/backup.c "
            f"source-sharding scheme; {'start-4' if workload == 'config2' else 'the first rows of start-111'}); "
            "a CPU visit relaxes both directions of an edge")


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    workload = args.workload if args.workload in ("config2", "config3") else "config3"
    step_s, step_v, kind, cores = cpu_reference_run(args.steps, args.warmup, workload)
    total_s, total_v = sum(step_s), sum(step_v)
    value = total_v / total_s / 1e9
    line = {
        "impl": "reference", "metric": "GRelax/s", "value": value, "unit": "GRelax/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total_s / args.steps,
        "higher_is_better": True, "scaling": "weak" if workload == "config2" else "strong", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOADS[workload],
                   "note": "CPU reference on ALL host cores whatever --gpus is: (node, offset) visits of serial_new "
                           "sweepXYZ, each visit relaxes both directions of the edge"},
        "cpu_baseline": {"value": value, "unit": "GRelax/s", "cores": cores, "kind": kind,
                         "sample": cpu_sample_text(cores, workload)},
        "e2e": {"value": value, "unit": "GRelax/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    sweeps = _ref_sweeps_per_source()
    if sweeps:   # converged sources/s: measured visit rate / (visits per sweep x the reference's recorded sweep counts)
        mean = sum(sweeps) / len(sweeps)
        line["converged_sources_per_s"] = value * 1e9 / (VISITS_PER_SWEEP_818 * mean)
        line["config"]["sources_per_s_note"] = (
            f"extrapolated: measured visits/s over {mean:.1f} sweeps per source (mean of the {len(sweeps)} converged "
            "reference runs recorded in tests/golden/*.json)")
    print(json.dumps(line), flush=True)
    return 0


def kernel_code_sha256():
    """sha256 of csrc/kernels.cu with comments and white space removed (a comment edit does not stale the capture)."""
    src = (ROOT / "uoparallel_seismic_project_b200" / "csrc" / "kernels.cu").read_text()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    src = re.sub(r"//[^\n]*", "", src)
    return hashlib.sha256("".join(src.split()).encode()).hexdigest()


def _ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel from the committed ncu --set full
    capture -- only while csrc/kernels.cu is still the code that was profiled (else the number is stale: None)."""
    try:
        t = json.loads((ROOT / "profiles" / "r02_traffic.json").read_text())
        if t.get("kernels_cu_code_sha256") != kernel_code_sha256():
            return None, f"stale: {t.get('source')} was taken with another kernels.cu"
        return t["dram_bytes_per_launch"], t["source"]
    except Exception:
        return None, None


def _golden(label):
    for name in ("full_241.json", "full_241_more.json"):
        try:
            for g in json.loads((ROOT / "tests" / "golden" / name).read_text()):
                if g["label"] == label:
                    return g
        except Exception:
            pass
    return None


# ------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------
def dump_outputs(ctx, nsrc, dims, out_dir, name):
    """Travel times of the context's last solve as out_dir/<name>.npy, float32[nsrc, DUMP_NODES]: row s holds source s's
    field at DUMP_NODES flat node indices drawn without replacement by numpy's default_rng(0) and sorted -- the same
    nodes for every source and every run.  (The full fields of config 3 are 1.3 GB.)"""
    import numpy as np
    n = int(np.prod(dims))
    idx = np.sort(np.random.default_rng(0).choice(n, size=min(n, DUMP_NODES), replace=False))
    field = np.empty(dims, np.float32)
    out = np.empty((nsrc, len(idx)), np.float32)
    for s in range(nsrc):
        out[s] = ctx.get_tt(s, out=field).ravel()[idx]
    d = pathlib.Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    np.save(d / f"{name}.npy", out)


def timed_resident(P, torch, ctx, stream, flush, steps, warmup, barrier, before_timed=None):
    """W untimed + K timed device-resident solves (CUDA events on the solve stream, L2 flushed in between)."""
    for _ in range(warmup):
        ctx.run()
    if before_timed:
        before_timed()
    barrier()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    acc = dict(relaxations=0, launches=0, rounds=0, tiles=0, relax_launches=0, units=0)
    wall0 = time.perf_counter()
    for k in range(steps):
        flush.zero_()                      # L2 flush between timed iterations (not timed)
        ev[k][0].record(stream)
        st = ctx.run()
        ev[k][1].record(stream)
        acc["relaxations"] += st.relaxations; acc["launches"] += st.kernel_launches; acc["rounds"] += st.rounds
        acc["tiles"] += st.tile_visits; acc["relax_launches"] += st.relax_launches; acc["units"] += st.units_run
    barrier()
    acc["wall_ms"] = (time.perf_counter() - wall0) * 1e3
    acc["dev_ms"] = sum(a.elapsed_time(b) for a, b in ev)
    return acc


def kernel_roofline(P, v, star, starts, local, stream, flush, reps, sms, sm_max):
    """The relax kernel alone: same solve, every launch bracketed with CUDA events on its own stream."""
    pctx = P.SweepContext(device=local, profile_kernels=1)
    pctx.set_stream(stream.cuda_stream)
    pctx.set_model(v); pctx.set_star(star); pctx.set_sources(starts)
    pctx.run()
    k_ms = k_launch = k_relax = k_tiles = 0
    for _ in range(reps):
        flush.zero_()
        st = pctx.run()
        k_ms += st.relax_kernel_ms; k_launch += st.relax_launches; k_relax += st.relaxations; k_tiles += st.tile_visits
    pctx.close()
    lane_ops = 4 * k_relax / (k_ms * 1e-3) / 1e12               # Tlane-op/s of the relax kernel alone
    peak_ops = sms * 128 * sm_max * 1e6 / 1e12
    return dict(k_ms=k_ms, k_launch=k_launch, k_relax=k_relax, k_tiles=k_tiles, reps=reps, lane_ops=lane_ops,
                peak_ops=peak_ops)


def extras_single_gpu(P, torch, W, local, stream, flush, sms, sm_max):
    """N=1 riders (short): BASELINE config 2 (start-4, 818-FS), config 1 (constant box, 3-FS, start-1) and the 5-FS
    star, each device-resident with its own relax-kernel roofline fraction."""
    out = {}
    cases = [("config2_818_start4", W.heterogeneous_field(DIMS, 7), "818", W.starts(4)),
             ("config1_const_3fs_start1", W.constant_field(DIMS), "3", W.starts(1)),
             ("hetero_5fs_start4", W.heterogeneous_field(DIMS, 7), "5", W.starts(4))]
    for name, v, starname, starts in cases:
        star = P.make_star(W.star(starname))
        ctx = P.SweepContext(device=local)
        ctx.set_stream(stream.cuda_stream)
        ctx.set_model(v); ctx.set_star(star); ctx.set_sources(starts)
        acc = timed_resident(P, torch, ctx, stream, flush, 5, 3, torch.cuda.synchronize)
        viol = sum(ctx.count_violations(s) for s in range(len(starts)))
        ctx.close()
        r = kernel_roofline(P, v, star, starts, local, stream, flush, 3, sms, sm_max)
        out[name] = {"ms_per_solve": acc["dev_ms"] / 5, "grelax_per_s": acc["relaxations"] / acc["dev_ms"] / 1e6,
                     "converged_sources_per_s": len(starts) * 5 / acc["dev_ms"] * 1e3,
                     "tile_visits_per_solve": acc["tiles"] / 5, "violations": viol,
                     "roofline_frac": r["lane_ops"] / r["peak_ops"], "relax_launches_per_solve": r["k_launch"] / r["reps"]}
    return out


def one_grid_rider(P, W, ndev):
    """ONE source on ONE 1201x1201x251 grid: all devices of the box against one device, same code path
    (sweeptt_solve_slabs: shared box in peer memory, halo reads fused into the relaxation kernel's TMA loads)."""
    dims = (1201, 1201, 251)
    v = W.heterogeneous_field(dims, 11)
    star = P.make_star(W.star("818"))
    start = (600, 600, 250)
    out = {"workload": "1201x1201x251 heterogeneous (seed 11), 818-FS, 1 source at (600,600,250)", "devices": ndev}
    sha = {}
    for n in (1, ndev):
        best = None
        for _ in range(2):
            tt, st = P.solve_slabs(v, star, start, num_slabs=n, slab_axis=0)
            if best is None or st.solve_ms < best.solve_ms:
                best = st
        sha[n] = hashlib.sha256(tt.tobytes()).hexdigest()
        out[f"solve_ms_{n}_dev"] = best.solve_ms
        out[f"grelax_per_s_{n}_dev"] = best.relaxations / best.solve_ms / 1e6
        out[f"devices_used_{n}"] = best.devices_used
        del tt
    out["speedup"] = out["solve_ms_1_dev"] / out[f"solve_ms_{ndev}_dev"]
    out["bit_equal_to_one_device"] = sha[1] == sha[ndev]
    out["sha256"] = sha[ndev]
    return out


def run_ours(args):
    import numpy as np
    import torch
    import uoparallel_seismic_project_b200 as P
    from uoparallel_seismic_project_b200 import api, dispatch, workloads as W

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the sweep has no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    dims = DIMS
    scaling = "strong"
    src_ids = None
    if args.workload == "config2":
        v = W.heterogeneous_field(dims, 7)
        starts = dispatch.sources_for_rank(rank, world)
        scaling = "weak"
    elif args.workload == "config3":
        v = W.heterogeneous_field(dims, 7)
        src_ids = dispatch.shard_round_robin(111, rank, world)
        starts = W.starts(111)[src_ids]
    else:
        dims = (1201, 1201, 251)
        v = W.heterogeneous_field(dims, 11)
        starts = (W.starts(24) * 5)[dispatch.shard_round_robin(24, rank, world)]
    workload = WORKLOADS[args.workload]
    star = P.make_star(W.star("818"))
    nsrc = len(starts)
    props = torch.cuda.get_device_properties(local)
    sms = props.multi_processor_count
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    # ---- device-resident leg: slowness + star + sources already in HBM -------------------------
    stream = torch.cuda.Stream(device=dev)   # not the legacy default stream: the solver captures CUDA graphs on it
    torch.cuda.set_stream(stream)
    ctx = P.SweepContext(device=local)
    ctx.set_stream(stream.cuda_stream)
    ctx.set_model(v); ctx.set_star(star); ctx.set_sources(starts)
    box = {}
    acc = timed_resident(P, torch, ctx, stream, flush, args.steps, args.warmup, barrier,
                         before_timed=lambda: box.setdefault("sampler", ClockSampler(local) if rank == 0 else None))
    clocks = box["sampler"].stop() if box.get("sampler") else None
    if args.dump_outputs:
        dump_outputs(ctx, nsrc, dims, args.dump_outputs, "tt" if world == 1 else f"tt_rank{rank}")
    tot = dispatch.combine(dist, dev, elapsed_ms=acc["dev_ms"], relaxations=acc["relaxations"],
                           sources=nsrc * args.steps, launches=acc["launches"])
    pulls_per_grid_round = ctx.relaxations_per_round   # in-bounds pulls of ONE full round of one source (analytic)
    # ---- parity riders: every rank's fields are fixed points; source 0 against the reference's own hash ----
    viol = sum(ctx.count_violations(s) for s in range(nsrc))
    viol_all = dispatch.combine(dist, dev, elapsed_ms=0.0, relaxations=viol, sources=0, launches=0)["relaxations"]
    parity = {"fixed_point_violations_all_ranks": int(viol_all)}
    if rank == 0 and args.workload in ("config2", "config3"):
        tt0 = ctx.get_tt(0)
        parity["source0_sha256"] = hashlib.sha256(tt0.tobytes()).hexdigest()
        g = _golden("config3_hetero_818_row0" if args.workload == "config3" else "config2_hetero_818_src0")
        parity["source0_matches_reference_sha256"] = (g["tt_sha256"] == parity["source0_sha256"]) if g else None
    assert viol_all == 0, "solve did not reach the fixed point"

    peaks = {}
    try:
        peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text())
    except OSError:
        pass
    sm_max = (clocks or {}).get("sm_max_mhz") or peaks.get("sm_max_mhz") or 1965.0
    sm_run = (clocks or {}).get("sm_mhz") or sm_max

    # ---- roofline of the dominant kernel (relax_tiled): same steps, every launch event-bracketed --
    roof = kernel_roofline(P, v, star, starts, local, stream, flush, max(1, min(args.steps, 5)), sms, sm_max)
    if args.workload == "config4":   # 24 x 1.45 GB of pinned host boxes: the extra workload reports the resident leg only
        ctx.close()
        if rank == 0:
            value = tot["relaxations"] / tot["elapsed_ms"] / 1e6
            print(json.dumps({"metric": "GRelax/s", "value": value, "unit": "GRelax/s", "n_gpus": world, "steps": args.steps,
                              "warmup": args.warmup, "ms_per_step": tot["elapsed_ms"] / args.steps, "higher_is_better": True,
                              "scaling": scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                              "config": {"workload": workload}, "converged_sources_per_s": tot["sources"] / tot["elapsed_ms"] * 1e3,
                              "clocks": clocks, "gpu_launches": tot["launches"], "e2e": None, "parity": parity,
                              "roofline": {"bound": "fp32-issue", "kernel": "relax_tiled<7, fs818>", "unit": "TFLOP/s",
                                           "achieved": roof["lane_ops"], "peak": roof["peak_ops"],
                                           "frac": roof["lane_ops"] / roof["peak_ops"]}}), flush=True)
        if dist is not None:
            dist.destroy_process_group()
        return 0

    # ---- end-to-end leg: pinned host buffers through the one-shot C-ABI call ----------------------
    hv = torch.from_numpy(v).pin_memory()
    hout = torch.empty((nsrc,) + dims, dtype=torch.float32).pin_memory()
    st_arr = api._make_starts(starts)
    ptrs = (ctypes.c_void_p * nsrc)(*[hout[s].data_ptr() for s in range(nsrc)])
    opts = api._opts(device=local)
    for _ in range(args.warmup):
        api.solve_raw(hv.data_ptr(), dims, star, st_arr, ptrs, opts)
    barrier()
    e2e_relax = 0
    d2h_tail_ms = 0.0
    t0 = time.perf_counter()
    for _ in range(args.steps):
        s2 = api.solve_raw(hv.data_ptr(), dims, star, st_arr, ptrs, opts)
        e2e_relax += s2.relaxations
        d2h_tail_ms += s2.d2h_ms
    barrier()
    e2e_ms = (time.perf_counter() - t0) * 1e3
    e2e = dispatch.combine(dist, dev, elapsed_ms=e2e_ms, relaxations=e2e_relax, sources=nsrc * args.steps, launches=0)
    if rank == 0:
        got = hout[0].numpy()
        assert np.array_equal(got.view(np.uint32), ctx.get_tt(0).view(np.uint32)), "e2e and resident legs disagree"
    ctx.close()
    P.load_library().sweeptt_release_cache()
    del hout

    # ---- N>1 rider: ONE grid spread over all N devices (config 5's scheme at config 4's size), driven by rank 0 ----
    one_grid = None
    if world > 1 and not args.no_extras and args.workload == "config3":
        host_group = dist.new_group(backend="gloo")     # host-side wait: no NCCL kernel spins on the devices meanwhile
        if rank == 0:
            try:
                one_grid = one_grid_rider(P, W, world)
            except Exception as e:  # a rider must never sink the headline
                one_grid = {"failed": repr(e)}
        dist.barrier(group=host_group)

    extras = None
    if rank == 0 and world == 1 and not args.no_extras and args.workload == "config3":
        try:
            extras = extras_single_gpu(P, torch, W, local, stream, flush, sms, sm_max)
        except Exception as e:  # a rider must never sink the headline
            extras = {"failed": repr(e)}

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return 0

    value = tot["relaxations"] / tot["elapsed_ms"] / 1e6          # GRelax/s, whole job
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    tile_bytes = 8 * 8 * 8 * 12                                 # algorithmic bytes per tile visit (8x8x8 nodes x 12 B)
    launches_per_step = roof["k_launch"] / roof["reps"]
    alg_bytes_per_launch = tile_bytes * roof["k_tiles"] / max(1, roof["k_launch"])
    hbm_achieved = tile_bytes * roof["k_tiles"] / (roof["k_ms"] * 1e-3) / 1e9 if roof["k_ms"] else None
    traffic, traffic_src = _ncu_traffic() if args.workload == "config3" else (None, None)
    line = {
        "metric": "GRelax/s", "value": value, "unit": "GRelax/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": tot["elapsed_ms"] / args.steps, "higher_is_better": True,
        "scaling": scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload, "sources_total": tot["sources"] // args.steps, "sources_on_rank0": nsrc,
                   "loop": (f"{launches_per_step:.0f} single persistent launches per solve (waves of <= 8 sources back to back; "
                            "work lists built on the device)" if launches_per_step <= 64
                            else "CUDA-graph WHILE of rounds (device-resident)"),
                   "l2": "flushed between timed steps (512 MiB write, untimed)",
                   "relax_definition": "one pull evaluation tt[n] <- min(tt[n], hd*(v_n+v_m)+tt[m]) with n,m in bounds"},
        "converged_sources_per_s": tot["sources"] / tot["elapsed_ms"] * 1e3,
        "rounds_per_step": acc["rounds"] / args.steps, "tile_visits_per_step": acc["tiles"] / args.steps,
        "pulls_per_source": tot["relaxations"] / max(1, tot["sources"]),
        "grid_equivalents_per_source": tot["relaxations"] / max(1, tot["sources"]) / pulls_per_grid_round,
        "wall_ms_timed_region": acc["wall_ms"],
        "clocks": clocks,
        "gpu_launches": tot["launches"],
        "parity": parity,
        "e2e": {"value": e2e["relaxations"] / e2e["elapsed_ms"] / 1e6, "unit": "GRelax/s",
                "converged_sources_per_s": e2e["sources"] / e2e["elapsed_ms"] * 1e3,
                "ms_per_step": e2e["elapsed_ms"] / args.steps,
                "timing": "host wall clock around sweeptt_solve() (H2D of the model, solve, D2H of every field; the "
                          "copies of finished waves run behind the solve of the next ones)",
                "d2h_tail_ms_per_step_rank0": d2h_tail_ms / args.steps,
                "h2d_bytes_per_step": int(np.prod(dims)) * 4 * world,
                "d2h_bytes_per_step": int(np.prod(dims)) * 4 * (tot["sources"] // args.steps)},
        "roofline": {
            "bound": "fp32-issue", "kernel": "relax_tiled<7, fs818>",
            "achieved": roof["lane_ops"], "peak": roof["peak_ops"], "unit": "TFLOP/s", "frac": roof["lane_ops"] / roof["peak_ops"],
            "frac_at_run_clock": roof["lane_ops"] / (sms * 128 * sm_run * 1e6 / 1e12),
            "grelax_per_s_kernel": roof["k_relax"] / (roof["k_ms"] * 1e-3) / 1e9,
            "avg_launch_ms": roof["k_ms"] / max(1, roof["k_launch"]), "launches_measured": roof["k_launch"],
            "peak_source": f"{sms} SMs x 128 lanes x {sm_max:.0f} MHz (clocks.max.sm), 4 fp32 operations per pull "
                           "(FADD, FMUL, FADD, FMNMX; no FMA allowed by the bit-exactness contract)",
            "hbm": {"achieved": hbm_achieved, "peak": hbm_peak, "unit": "GB/s",
                    "frac": hbm_achieved / hbm_peak if hbm_achieved else None,
                    "note": "12 B per node per tile visit; the path is ~50x away from the HBM roof (SURVEY.md 8d)"},
            # executed but not counted: lanes of partly filled edge tiles and pulls across the box boundary
            # (241 = 30 tiles + 1 node along two axes): counted pulls / (unit visits x 256 nodes x 817 pull offsets)
            "counted_over_executed_lane_pulls": acc["relaxations"] / max(1, acc["units"] * 256 * 817),
            "frac_of_executed_lane_pulls": (roof["lane_ops"] / roof["peak_ops"]) / max(1e-9, acc["relaxations"] / max(1, acc["units"] * 256 * 817)),
            "traffic": traffic, "traffic_source": traffic_src,
            "algorithmic_bytes_per_launch": alg_bytes_per_launch,
        },
    }
    try:   # the reference's OWN CUDA programs timed on a B200 of this pool (tools/legacy_gpu.py; a cited measurement)
        lg = json.loads((ROOT / "profiles" / "r02_legacy_gpu.json").read_text())
        line["legacy_gpu"] = {
            "source": "profiles/r02_legacy_gpu.json (tools/legacy_gpu.py: cuda/cudasweep-tt-multistart_230.cu and _380.cu compiled "
                      "unmodified with nvcc -arch=sm_100, config 2, same pool's B200; not re-run inside bench.py)",
            "ms_per_converged_source": {k: v.get("ms_per_converged_source_mean") for k, v in lg["variants"].items()},
            "kernel_ms_per_sweep": {k: v.get("kernel_ms_per_sweep_mean") for k, v in lg["variants"].items()},
            "sweeps_per_source": {k: v.get("sweeps_per_source") for k, v in lg["variants"].items()},
            "output_tt_equals_ours": {k: v.get("output_tt_equals_ours") for k, v in lg["variants"].items()},
            "ours_ms_per_converged_source_per_gpu": tot["elapsed_ms"] * world / max(1, tot["sources"]),
        }
    except Exception:
        pass
    if extras is not None:
        line["extras"] = extras
    if one_grid is not None:
        line["one_grid_over_all_gpus"] = one_grid
    if not args.no_cpu_baseline and world == 1 and args.workload in ("config2", "config3"):
        try:
            step_s, step_v, kind, cores = cpu_reference_run(2, 1, args.workload)
            line["cpu_baseline"] = {"value": sum(step_v) / sum(step_s) / 1e9, "unit": "GRelax/s", "cores": cores,
                                    "kind": kind, "sample": "2 timed + 1 warm-up steps; " + cpu_sample_text(cores, args.workload)}
        except Exception as e:  # the baseline must never sink the GPU number
            line["cpu_baseline"] = {"value": None, "unit": "GRelax/s", "cores": 0, "kind": "port", "sample": f"failed: {e}"}
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    a = parse()
    sys.exit(run_reference(a) if a.impl == "reference" else run_ours(a))
