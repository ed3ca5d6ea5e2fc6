#!/usr/bin/env python3
"""Generate tests/golden/* from the REFERENCE ITSELF (oracle/_ref = unmodified
serial_new/sweep-tt-multistart.c compiled in the build container).

  python tools/make_golden.py small     -> tests/golden/small_cases.npz   (seconds)
  python tools/make_golden.py full      -> tests/golden/full_241.json     (~15-25 min, 5 processes)
  python tools/make_golden.py config3_all [P] -> tests/golden/config3_all.json (every other row of start-111, sha256 only)
  python tools/make_golden.py more [P]  -> tests/golden/full_241_more.json (round 2: 9 further config-3 sources,
                                           full-size 5-FS and a scaled config-4-like box; P processes, ~1 h on 6)
  python tools/make_golden.py pins      -> tests/golden/oracle_pins.json (see pins(); needs no reference)

The GPU box has no /root/reference; the parity tests there compare against these files.
Small cases: converged float32 fields for seeded boxes.  Full size (BASELINE configs 1 and 2):
sha256 of the converged field + every 4999th float + the reference's sweep count.
"""
import hashlib
import json
import multiprocessing as mp
import pathlib
import sys
import time

import numpy as np

ROOT = pathlib.Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
import oracle  # noqa: E402
from uoparallel_seismic_project_b200 import workloads as W  # noqa: E402

GOLD = ROOT / "tests" / "golden"

SMALL = [
    # name, dims, field kind, seed, star, starts
    ("rand_3fs", (12, 11, 9), "random", 1, "3", [(5, 5, 4), (0, 0, 0), (11, 10, 8)]),
    ("rand_5fs", (12, 11, 9), "random", 2, "5", [(6, 2, 8), (0, 10, 0)]),
    ("rand_818", (12, 11, 9), "random", 3, "818", [(5, 5, 4), (11, 0, 8)]),
    ("const_818", (20, 17, 13), "constant", 0, "818", [(10, 8, 12), (12, 9, 11), (0, 0, 0)]),
    ("hetero_818", (33, 25, 40), "hetero", 5, "818", [(16, 12, 39), (8, 8, 0), (32, 24, 39)]),
    ("contrast_5fs", (24, 24, 35), "contrast", 6, "5", [(3, 20, 17), (23, 23, 34)]),
    ("tileedge_818", (17, 16, 33), "random", 7, "818", [(8, 8, 32), (16, 15, 31), (7, 8, 0)]),
]


def field(kind, dims, seed):
    if kind == "random":
        return W.random_field(dims, seed)
    if kind == "constant":
        return W.constant_field(dims, 0.25)
    if kind == "hetero":
        return W.heterogeneous_field(dims, seed)
    if kind == "contrast":
        return W.contrast_field(dims, seed)
    raise ValueError(kind)


def small():
    out = {}
    meta = []
    for name, dims, kind, seed, star, starts in SMALL:
        v = field(kind, dims, seed)
        off = W.star(star)
        for si, st in enumerate(starts):
            tt, sweeps = oracle.ref_solve(v, off, st)
            out[f"{name}__{si}"] = tt
            meta.append(dict(case=name, idx=si, dims=dims, kind=kind, seed=seed, star=star, start=st, ref_sweeps=sweeps))
            print(name, st, "sweeps", sweeps)
        out[f"{name}__v_sha"] = np.frombuffer(hashlib.sha256(v.tobytes()).digest(), np.uint8)
    out["meta_json"] = np.frombuffer(json.dumps(meta).encode(), np.uint8)
    np.savez_compressed(GOLD / "small_cases.npz", **out)


def _full_one(job):
    label, kind, seed, star, start = job[:5]
    dims = tuple(job[5]) if len(job) > 5 else (241, 241, 51)
    v = field(kind, dims, seed)
    t0 = time.time()
    tt, sweeps = oracle.ref_solve(v, W.star(star), start)
    flat = tt.ravel()
    return dict(label=label, kind=kind, seed=seed, star=star, start=list(map(int, start)), dims=list(dims), ref_sweeps=sweeps,
                seconds=round(time.time() - t0, 1), v_sha256=hashlib.sha256(v.tobytes()).hexdigest(),
                tt_sha256=hashlib.sha256(tt.tobytes()).hexdigest(), sample_stride=4999,
                sample_bits=[int(x) for x in flat[::4999].view(np.uint32)])


def full():
    jobs = [("config1_const_3fs", "constant", 0, "3", tuple(W.starts(1)[0]))]
    for s, st in enumerate(W.starts(4)):
        jobs.append((f"config2_hetero_818_src{s}", "hetero", 7, "818", tuple(st)))
    with mp.Pool(len(jobs)) as pool:
        res = pool.map(_full_one, jobs)
    (GOLD / "full_241.json").write_text(json.dumps(res, indent=1))
    for r in res:
        print(r["label"], r["ref_sweeps"], r["seconds"], r["tt_sha256"][:16])


MORE_C3 = [0, 13, 27, 41, 55, 69, 83, 97, 110]          # rows of docs/start-111-241-241-51.txt
C4_DIMS = (301, 301, 64)                                 # scaled config-4-like box (seed 11 like config 4)
C4_STARTS = [(15, 25, 63), (150, 150, 63), (285, 40, 63), (60, 270, 63), (240, 240, 63), (150, 20, 63)]


def more():
    procs = int(sys.argv[2]) if len(sys.argv) > 2 else 6
    jobs = []
    s111 = W.starts(111)
    for i in MORE_C3:
        jobs.append((f"config3_hetero_818_row{i}", "hetero", 7, "818", tuple(int(c) for c in s111[i])))
    jobs.append(("full_hetero_5fs_start1", "hetero", 7, "5", tuple(int(c) for c in W.starts(1)[0])))
    jobs.append(("full_const_5fs_start1", "constant", 0, "5", tuple(int(c) for c in W.starts(1)[0])))
    for s, st in enumerate(C4_STARTS):
        jobs.append((f"config4like_hetero_818_src{s}", "hetero", 11, "818", st, C4_DIMS))
    out = GOLD / "full_241_more.json"
    res = []
    with mp.Pool(procs) as pool:
        for r in pool.imap_unordered(_full_one, jobs):
            res.append(r)
            res.sort(key=lambda x: x["label"])
            out.write_text(json.dumps(res, indent=1))     # partial results survive an interrupted run
            print(r["label"], r["ref_sweeps"], r["seconds"], r["tt_sha256"][:16], flush=True)


def _sha_only(job):
    r = _full_one(job)
    r.pop("sample_bits", None); r.pop("sample_stride", None)
    return r


def config3_all():
    """Every row of docs/start-111 that full_241_more.json does not hold yet: sha256 + sweep count only (0.3 KB each),
    into tests/golden/config3_all.json -- ~15 min per source per core."""
    procs = int(sys.argv[2]) if len(sys.argv) > 2 else 7
    s111 = W.starts(111)
    out = GOLD / "config3_all.json"
    res = json.loads(out.read_text()) if out.exists() else []
    have = {r["label"] for r in res}
    jobs = [(f"config3_hetero_818_row{i}", "hetero", 7, "818", tuple(int(c) for c in s111[i]))
            for i in range(111) if i not in MORE_C3 and f"config3_hetero_818_row{i}" not in have]
    with mp.Pool(procs) as pool:
        for r in pool.imap_unordered(_sha_only, jobs):
            res.append(r)
            res.sort(key=lambda x: int(x["label"].rsplit("row", 1)[1]))
            out.write_text(json.dumps(res, indent=0))
            print(r["label"], r["ref_sweeps"], r["seconds"], r["tt_sha256"][:16], flush=True)


PIN_TRACE = dict(kind="contrast", dims=(14, 13, 12), seed=4, start=(7, 3, 11))


def pin_vbox_bytes(tmp):
    """The .vbox files of the cases tests/test_formats.py compares with the reference's own tools and loaders."""
    import subprocess
    import uoparallel_seismic_project_b200 as P
    tmp = pathlib.Path(tmp)
    out = {}
    P.vbox_store(tmp / "a.vbox", (W.random_field((7, 5, 9), seed=3) - np.float32(0.25)).astype(np.float32), origin=(1, 1, 1))
    out["vbox_store_random_7x5x9_seed3_minus_quarter"] = (tmp / "a.vbox").read_bytes()
    W.write_text_a(tmp / "v.txt", W.heterogeneous_field((5, 6, 7), seed=9))
    subprocess.run([str(P.lib_path().parent / "vconvert"), str(tmp / "v.txt"), str(tmp / "b.vbox")], check=True,
                   capture_output=True)
    out["vconvert_hetero_5x6x7_seed9"] = (tmp / "b.vbox").read_bytes()
    P.vbox_store(tmp / "c.vbox", W.random_field((5, 4, 6), seed=8), origin=(1, 1, 1))
    out["vbox_store_random_5x4x6_seed8"] = (tmp / "c.vbox").read_bytes()
    return {k: hashlib.sha256(v).hexdigest() for k, v in out.items()}


def restatement_trace(star):
    """(stores, sha256 of the field) after every sweep of the restatement on the PIN_TRACE case, up to the first sweep
    that stores nothing -- the sequence oracle.ref_solve(per_sweep=...) yields for the reference's own sweepXYZ."""
    v = field(PIN_TRACE["kind"], PIN_TRACE["dims"], PIN_TRACE["seed"])
    off = W.star(star)
    tt = oracle.init_tt(v.shape, PIN_TRACE["start"])
    trace = []
    while True:
        c = oracle.sweep(v, tt, off, PIN_TRACE["start"])
        trace.append((int(c), hashlib.sha256(tt.tobytes()).hexdigest()))
        if c == 0:
            return trace


def pins():
    """tests/golden/oracle_pins.json: the quantities the CPU tests compare with the original project's own code when a
    checkout of it is at hand (SWEEPTT_REFERENCE) -- star distances, the per-sweep trace of the restatement, .vbox bytes --
    recorded from the restatement and this project's writers, so that the comparison also runs without the checkout."""
    import tempfile
    stars = ("3", "5", "818")
    with tempfile.TemporaryDirectory() as tmp:
        vbox = pin_vbox_bytes(tmp)
    res = {
        "provenance": "recorded by tools/make_golden.py pins from oracle/sweep_oracle.c and the project's .vbox writers; "
                      "tests/test_oracle.py and tests/test_formats.py compare the same quantities with the original "
                      "project's own code when SWEEPTT_REFERENCE names a checkout of it",
        "star_distance_bits": {s: [int(x) for x in oracle.star_distances(W.star(s)).view(np.uint32)] for s in stars},
        "trace_case": {k: list(v) if isinstance(v, tuple) else v for k, v in PIN_TRACE.items()},
        "trace": {s: [list(t) for t in restatement_trace(s)] for s in stars},
        "vbox_sha256": vbox,
    }
    (GOLD / "oracle_pins.json").write_text(json.dumps(res, indent=0) + "\n")


if __name__ == "__main__":
    {"small": small, "full": full, "more": more, "config3_all": config3_all, "pins": pins}[sys.argv[1]]()
