"""ctypes binding of include/sweeptt.h -- the reference-facing call surface.

Names follow the reference: ``FS`` / ``START`` are the structs of
serial_new/sweep-tt-multistart.c:46-58; :func:`solve` stands where ``cudaRun`` /
the ``while(anychange) sweepXYZ`` loop stood (cuda/cudasweep-tt-multistart.cu:227,
serial_new/...c:150-170); boxes are FLOATBOX-ordered ``float32[nx, ny, nz]`` (z fastest,
include/floatbox.h:127-129).  Error behaviour mirrors the ABI: a zero return becomes a
:class:`SweepError` carrying ``sweeptt_last_error()``.
"""
from __future__ import annotations

import ctypes as C
import os
import pathlib
import weakref
from dataclasses import dataclass

import numpy as np

_PKG = pathlib.Path(__file__).resolve().parent
_LIB = None

KERNEL_AUTO, KERNEL_SIMPLE, KERNEL_TILED = 0, 1, 2
LOOP_AUTO, LOOP_BATCHED, LOOP_GRAPH = 0, 1, 2
# status of a traced ray (SWEEPTT_RAY_*, include/sweeptt.h)
RAY_OK, RAY_UNREACHED, RAY_NOT_FIXED_POINT, RAY_NO_PREDECESSOR, RAY_STALLED, RAY_TRUNCATED = range(6)
# status of a located event (SWEEPTT_LOC_*, include/sweeptt.h)
LOC_OK, LOC_NO_PICKS, LOC_UNREACHED = range(3)


class SweepError(RuntimeError):
    pass


class FS(C.Structure):
    _fields_ = [("i", C.c_int), ("j", C.c_int), ("k", C.c_int), ("d", C.c_float)]


class START(C.Structure):
    _fields_ = [("i", C.c_int), ("j", C.c_int), ("k", C.c_int)]


class _Opts(C.Structure):
    _fields_ = [
        ("struct_size", C.c_int), ("device", C.c_int), ("num_devices", C.c_int), ("kernel", C.c_int),
        ("loop", C.c_int), ("rounds_per_poll", C.c_int), ("max_rounds", C.c_int), ("star_used", C.c_int),
        ("verbose", C.c_int), ("slab_axis", C.c_int), ("profile_kernels", C.c_int),
    ]


class _Stats(C.Structure):
    _fields_ = [
        ("struct_size", C.c_int), ("rounds", C.c_int), ("kernel_used", C.c_int), ("devices_used", C.c_int),
        ("kernel_launches", C.c_longlong), ("tile_visits", C.c_longlong), ("relaxations", C.c_longlong),
        ("solve_ms", C.c_double), ("relax_kernel_ms", C.c_double), ("relax_launches", C.c_longlong),
        ("h2d_ms", C.c_double), ("d2h_ms", C.c_double), ("h2d_bytes", C.c_longlong), ("d2h_bytes", C.c_longlong),
        ("units_run", C.c_longlong), ("units_changed", C.c_longlong),
    ]


class _LsqrOpts(C.Structure):
    _fields_ = [("struct_size", C.c_int), ("damp", C.c_double), ("smooth", C.c_double), ("atol", C.c_double),
                ("btol", C.c_double), ("conlim", C.c_double), ("iter_lim", C.c_int)]


class _LsqrInfo(C.Structure):
    _fields_ = [("struct_size", C.c_int), ("istop", C.c_int), ("itn", C.c_int), ("r1norm", C.c_double),
                ("r2norm", C.c_double), ("anorm", C.c_double), ("acond", C.c_double), ("arnorm", C.c_double),
                ("xnorm", C.c_double)]


@dataclass
class SweepStats:
    rounds: int = 0
    kernel_used: int = 0
    devices_used: int = 0
    kernel_launches: int = 0
    tile_visits: int = 0
    relaxations: int = 0
    solve_ms: float = 0.0
    relax_kernel_ms: float = 0.0
    relax_launches: int = 0
    h2d_ms: float = 0.0
    d2h_ms: float = 0.0
    h2d_bytes: int = 0
    d2h_bytes: int = 0
    units_run: int = 0
    units_changed: int = 0

    @classmethod
    def _from(cls, s: _Stats) -> "SweepStats":
        return cls(**{f: getattr(s, f) for f in cls.__dataclass_fields__})


def lib_path() -> pathlib.Path:
    import os
    if os.environ.get("SWEEPTT_LIB"):  # developer override: an experimental build of the same ABI
        return pathlib.Path(os.environ["SWEEPTT_LIB"])
    return _PKG / "lib" / "libsweeptt.so"


_EXPORTS = [
    "sweeptt_device_count", "sweeptt_device_info", "sweeptt_last_error", "sweeptt_version",
    "sweeptt_star_fill_distances", "sweeptt_build_pull_star", "sweeptt_debug_column_split", "sweeptt_solve", "sweeptt_release_cache",
    "sweeptt_host_alloc", "sweeptt_host_free",
    "sweeptt_create", "sweeptt_destroy", "sweeptt_set_stream", "sweeptt_set_model", "sweeptt_set_star",
    "sweeptt_set_sources", "sweeptt_run", "sweeptt_step", "sweeptt_reset", "sweeptt_get_tt", "sweeptt_put_tt",
    "sweeptt_count_violations", "sweeptt_trace_rays", "sweeptt_ray_project", "sweeptt_ray_backproject",
    "sweeptt_rayset_freeze", "sweeptt_rayset_destroy", "sweeptt_rayset_bytes", "sweeptt_rayset_table",
    "sweeptt_rayset_paths", "sweeptt_rayset_project", "sweeptt_rayset_backproject", "sweeptt_rayset_lsqr",
    "sweeptt_locate_events", "sweeptt_misfit_regions",
    "sweeptt_misfit_box", "sweeptt_relaxations_per_round", "sweeptt_pool_bytes", "sweeptt_tiles_per_source", "sweeptt_debug_model_stats", "sweeptt_solve_slabs",
    "sweeptt_solve_slabs_vbox", "sweeptt_vbox_dims",
    "sweeptt_vbox_load", "sweeptt_vbox_store", "sweeptt_vbox_load_subset", "sweeptt_text_load",
    "sweeptt_star_load", "sweeptt_starts_load", "sweeptt_write_output_tt", "sweeptt_free",
]


def load_library() -> C.CDLL:
    """Load libsweeptt.so (never a fallback: a missing extension is an error)."""
    global _LIB
    if _LIB is not None:
        return _LIB
    p = lib_path()
    if not p.exists():
        raise SweepError(f"{p} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                         "(the sweep has no CPU fallback)")
    lib = C.CDLL(str(p))
    fp, ip = C.POINTER(C.c_float), C.POINTER(C.c_int)
    lib.sweeptt_last_error.restype = C.c_char_p
    lib.sweeptt_version.restype = C.c_char_p
    lib.sweeptt_device_info.argtypes = [C.c_int, C.c_char_p, C.c_int, ip, ip, C.POINTER(C.c_size_t)]
    lib.sweeptt_star_fill_distances.argtypes = [C.POINTER(FS), C.c_int, C.c_float]
    lib.sweeptt_star_fill_distances.restype = None
    lib.sweeptt_build_pull_star.argtypes = [C.POINTER(FS), C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
    lib.sweeptt_solve.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(FS), C.c_int, C.POINTER(START),
                                  C.c_int, C.POINTER(C.c_void_p), C.POINTER(_Opts), C.POINTER(_Stats)]
    lib.sweeptt_release_cache.restype = None
    lib.sweeptt_host_alloc.argtypes = [C.c_size_t]
    lib.sweeptt_host_alloc.restype = C.c_void_p
    lib.sweeptt_host_free.argtypes = [C.c_void_p]
    lib.sweeptt_host_free.restype = None
    lib.sweeptt_create.argtypes = [C.POINTER(_Opts)]
    lib.sweeptt_create.restype = C.c_void_p
    lib.sweeptt_destroy.argtypes = [C.c_void_p]
    lib.sweeptt_destroy.restype = None
    lib.sweeptt_set_stream.argtypes = [C.c_void_p, C.c_void_p]
    lib.sweeptt_set_model.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int]
    lib.sweeptt_set_star.argtypes = [C.c_void_p, C.POINTER(FS), C.c_int]
    lib.sweeptt_set_sources.argtypes = [C.c_void_p, C.POINTER(START), C.c_int]
    lib.sweeptt_run.argtypes = [C.c_void_p, C.POINTER(_Stats)]
    lib.sweeptt_step.argtypes = [C.c_void_p, C.c_int, ip, C.POINTER(_Stats)]
    lib.sweeptt_reset.argtypes = [C.c_void_p]
    lib.sweeptt_get_tt.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
    lib.sweeptt_put_tt.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
    lib.sweeptt_count_violations.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_longlong)]
    lib.sweeptt_trace_rays.argtypes = [C.c_void_p, C.c_int, C.c_int, C.POINTER(START), C.c_int, C.c_int, C.c_void_p,
                                       C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(_Stats)]
    lib.sweeptt_ray_project.argtypes = [C.c_void_p, C.c_int, C.c_int, C.POINTER(START), C.c_int, C.c_int, C.c_void_p,
                                        C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(_Stats)]
    lib.sweeptt_ray_backproject.argtypes = [C.c_void_p, C.c_int, C.c_int, C.POINTER(START), C.c_int, C.c_int,
                                            C.c_void_p, C.c_void_p, C.POINTER(C.c_int), C.c_void_p, C.POINTER(_Stats)]
    lib.sweeptt_rayset_freeze.argtypes = [C.c_void_p, C.c_int, C.c_int, C.POINTER(START), C.c_int, C.c_int,
                                          C.POINTER(_Stats)]
    lib.sweeptt_rayset_freeze.restype = C.c_void_p
    lib.sweeptt_rayset_destroy.argtypes = [C.c_void_p]
    lib.sweeptt_rayset_destroy.restype = None
    lib.sweeptt_rayset_bytes.argtypes = [C.c_void_p]
    lib.sweeptt_rayset_bytes.restype = C.c_size_t
    lib.sweeptt_rayset_table.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.sweeptt_rayset_paths.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    lib.sweeptt_rayset_project.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(_Stats)]
    lib.sweeptt_rayset_backproject.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_int),
                                               C.POINTER(_Stats)]
    lib.sweeptt_rayset_lsqr.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(_LsqrOpts), C.c_void_p,
                                        C.POINTER(_LsqrInfo), C.POINTER(_Stats)]
    lib.sweeptt_locate_events.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                          C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(_Stats)]
    lib.sweeptt_misfit_regions.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                           C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(_Stats)]
    lib.sweeptt_misfit_box.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.POINTER(_Stats)]
    lib.sweeptt_relaxations_per_round.argtypes = [C.c_void_p]
    lib.sweeptt_relaxations_per_round.restype = C.c_longlong
    lib.sweeptt_pool_bytes.argtypes = [C.c_void_p]
    lib.sweeptt_pool_bytes.restype = C.c_size_t
    lib.sweeptt_tiles_per_source.argtypes = [C.c_void_p]
    lib.sweeptt_tiles_per_source.restype = C.c_longlong
    lib.sweeptt_debug_model_stats.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.sweeptt_solve_slabs.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(FS), C.c_int, START,
                                        C.c_void_p, C.POINTER(_Opts), C.POINTER(_Stats)]
    lib.sweeptt_solve_slabs_vbox.argtypes = [C.c_char_p, C.POINTER(FS), C.c_int, START, C.c_void_p, C.POINTER(_Opts),
                                             C.POINTER(_Stats)]
    lib.sweeptt_vbox_dims.argtypes = [C.c_char_p, ip]
    lib.sweeptt_vbox_load.argtypes = [C.c_char_p, C.POINTER(fp), ip, ip]
    lib.sweeptt_vbox_store.argtypes = [C.c_char_p, C.c_void_p, ip, ip]
    lib.sweeptt_vbox_load_subset.argtypes = [C.c_char_p, ip, ip, C.POINTER(fp)]
    lib.sweeptt_text_load.argtypes = [C.c_char_p, C.POINTER(fp), ip, ip]
    lib.sweeptt_star_load.argtypes = [C.c_char_p, C.c_float, C.POINTER(C.POINTER(FS)), ip]
    lib.sweeptt_starts_load.argtypes = [C.c_char_p, C.POINTER(C.POINTER(START)), ip]
    lib.sweeptt_write_output_tt.argtypes = [C.c_char_p, C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_int, C.c_int]
    lib.sweeptt_free.argtypes = [C.c_void_p]
    lib.sweeptt_free.restype = None
    _LIB = lib
    return lib


def _check(ok, what: str):
    if not ok:
        raise SweepError(f"{what}: {load_library().sweeptt_last_error().decode()}")


def device_count() -> int:
    return load_library().sweeptt_device_count()


def make_star(offsets, delta: float = 10.0):
    """(L,3) int offsets -> FS[L] with d filled the reference's way (serial_new/...c:120-128)."""
    off = np.asarray(offsets, dtype=np.int32).reshape(-1, 3)
    arr = (FS * len(off))()
    for l, (a, b, c) in enumerate(off):
        arr[l].i, arr[l].j, arr[l].k = int(a), int(b), int(c)
    load_library().sweeptt_star_fill_distances(arr, len(off), C.c_float(delta))
    return arr


def _make_starts(starts):
    st = np.asarray(starts, dtype=np.int32).reshape(-1, 3)
    arr = (START * len(st))()
    for s, (a, b, c) in enumerate(st):
        arr[s].i, arr[s].j, arr[s].k = int(a), int(b), int(c)
    return arr


def _as_star(star, delta):
    return star if isinstance(star, C.Array) and star._type_ is FS else make_star(star, delta)


def _opts(**kw) -> _Opts:
    o = _Opts()
    o.struct_size = C.sizeof(_Opts)
    o.device = -1
    for k, v in kw.items():
        if v is not None:
            setattr(o, k, v)
    return o


def build_pull_star(star, star_used: int = 0, delta: float = 10.0):
    """Host-side edge-set analysis: (offsets int32[P,3], half distances f32[P], guard int32[P])."""
    fs = _as_star(star, delta)
    lib = load_library()
    cap = 2 * len(fs) + 4
    ijk = np.zeros((cap, 3), np.int32)
    hd = np.zeros(cap, np.float32)
    gd = np.zeros(cap, np.int32)
    n = lib.sweeptt_build_pull_star(fs, len(fs), star_used, ijk.ctypes.data, hd.ctypes.data, gd.ctypes.data, cap)
    if n < 0:
        raise SweepError("sweeptt_build_pull_star failed")
    return ijk[:n].copy(), hd[:n].copy(), gd[:n].copy()


def column_split(star, nw: int, delta: float = 10.0):
    """Test hook: (kmasks uint32[C], cuts uint16[6, G, nw+1]) -- how the tiled kernel shares the star's columns
    out between `nw` warps (six tables, see include/sweeptt.h)."""
    fs = _as_star(star, delta)
    lib = load_library()
    lib.sweeptt_debug_column_split.argtypes = [C.POINTER(FS), C.c_int, C.c_int, C.POINTER(C.c_int), C.c_void_p,
                                               C.c_int, C.c_void_p, C.c_int]
    lib.sweeptt_debug_column_split.restype = C.c_int
    cuts = np.zeros(6 * 64 * (nw + 1), np.uint16)
    kmasks = np.zeros(4096, np.uint32)
    ng = C.c_int(0)
    n = lib.sweeptt_debug_column_split(fs, len(fs), nw, C.byref(ng), cuts.ctypes.data, cuts.size, kmasks.ctypes.data,
                                       kmasks.size)
    if n < 0:
        raise SweepError("sweeptt_debug_column_split failed")
    return kmasks[:n].copy(), cuts[: 6 * ng.value * (nw + 1)].reshape(6, ng.value, nw + 1).copy()


def solve(slowness, star, starts, *, delta: float = 10.0, out=None, device: int | None = None,
          num_devices: int | None = None, kernel: int | None = None, loop: int | None = None,
          max_rounds: int | None = None, star_used: int | None = None, profile_kernels: int | None = None,
          rounds_per_poll: int | None = None, verbose: int | None = None):
    """One-shot multi-start solve with HOST buffers (the `cudaRun` replacement).

    slowness: float32[nx,ny,nz]; star: (L,3) offsets or FS array; starts: (S,3).
    Returns (tt float32[S,nx,ny,nz], SweepStats).  `out` may be a preallocated (pinned) array.
    """
    lib = load_library()
    v = np.ascontiguousarray(slowness, dtype=np.float32)
    if v.ndim != 3:
        raise SweepError("slowness must be a 3-D box")
    nx, ny, nz = v.shape
    fs = _as_star(star, delta)
    st = _make_starts(starts)
    ns = len(st)
    if out is None:
        out = np.empty((ns, nx, ny, nz), np.float32)
    if out.shape != (ns, nx, ny, nz) or out.dtype != np.float32 or not out.flags.c_contiguous:
        raise SweepError("out must be C-contiguous float32[S,nx,ny,nz]")
    ptrs = (C.c_void_p * ns)(*[out[s].ctypes.data for s in range(ns)])
    o = _opts(device=device, num_devices=num_devices, kernel=kernel, loop=loop, max_rounds=max_rounds,
              star_used=star_used, profile_kernels=profile_kernels, rounds_per_poll=rounds_per_poll, verbose=verbose)
    s = _Stats()
    _check(lib.sweeptt_solve(v.ctypes.data, nx, ny, nz, fs, len(fs), st, ns, ptrs, C.byref(o), C.byref(s)),
           "sweeptt_solve")
    return out, SweepStats._from(s)


def solve_slabs(slowness, star, start, *, num_slabs: int, slab_axis: int = 0, delta: float = 10.0,
                max_rounds: int | None = None, rounds_per_poll: int | None = None, verbose: int | None = None):
    """ONE source on ONE grid spread over `num_slabs` parts (the visible GPUs; more parts than GPUs share devices
    round-robin): the travel-time box is one range of peer memory whose pages are dealt block-cyclically along
    `slab_axis`, every part relaxes its own blocks and reads halo planes from the owner over NVLink inside the
    relaxation kernel -- no exchange step.  Replaces the MPI ghost-cell programs (mpi/16partsmpi.c:740-909).
    Returns (tt float32[nx,ny,nz], SweepStats)."""
    lib = load_library()
    v = np.ascontiguousarray(slowness, dtype=np.float32)
    nx, ny, nz = v.shape
    fs = _as_star(star, delta)
    st = START(int(start[0]), int(start[1]), int(start[2]))
    out = np.empty(v.shape, np.float32)
    o = _opts(num_devices=num_slabs, slab_axis=slab_axis, max_rounds=max_rounds, rounds_per_poll=rounds_per_poll,
              verbose=verbose)
    s = _Stats()
    _check(lib.sweeptt_solve_slabs(v.ctypes.data, nx, ny, nz, fs, len(fs), st, out.ctypes.data, C.byref(o), C.byref(s)),
           "sweeptt_solve_slabs")
    return out, SweepStats._from(s)


def solve_slabs_vbox(path, star, start, *, num_slabs: int, slab_axis: int = 0, delta: float = 10.0):
    """Like solve_slabs, but every part reads only the planes of its blocks from the .vbox file (subset loader)."""
    lib = load_library()
    d = (C.c_int * 3)()
    _check(lib.sweeptt_vbox_dims(os.fsencode(path), d), "sweeptt_vbox_dims")
    fs = _as_star(star, delta)
    st = START(int(start[0]), int(start[1]), int(start[2]))
    out = np.empty(tuple(d), np.float32)
    o = _opts(num_devices=num_slabs, slab_axis=slab_axis)
    s = _Stats()
    _check(lib.sweeptt_solve_slabs_vbox(os.fsencode(path), fs, len(fs), st, out.ctypes.data, C.byref(o), C.byref(s)),
           "sweeptt_solve_slabs_vbox")
    return out, SweepStats._from(s)


def solve_raw(v_ptr: int, dims, fs, starts_arr, out_ptrs, opts: _Opts):
    """Pointer-level call for bench.py's e2e leg (pinned torch tensors; no numpy in the way)."""
    lib = load_library()
    s = _Stats()
    _check(lib.sweeptt_solve(C.c_void_p(v_ptr), dims[0], dims[1], dims[2], fs, len(fs), starts_arr, len(starts_arr),
                             out_ptrs, C.byref(opts), C.byref(s)), "sweeptt_solve")
    return SweepStats._from(s)


@dataclass
class Rays:
    """Rays of sources [S] x receivers [R] (SweepContext.trace_rays).  nodes[s, r, :length[s, r]] are the ray's nodes
    (caller axes) from the receiver to the start; entries past the length are -1.  tt[s, r] = travel time at the
    receiver whatever the status (RAY_*)."""
    tt: np.ndarray        # float32[S, R]
    status: np.ndarray    # int32[S, R]
    length: np.ndarray    # int32[S, R]
    nodes: np.ndarray     # int32[S, R, max_nodes, 3]
    stats: SweepStats

    def path(self, s: int, r: int) -> np.ndarray:
        """int32[L, 3]: the nodes of ray (s, r), receiver first."""
        return self.nodes[s, r, : self.length[s, r]]


@dataclass
class RayProjection:
    """G*d over the rays of sources [S] x receivers [R] (SweepContext.ray_project): values[s, r] is the perturbation
    summed along the ray with the sweep's expression from the start towards the receiver (NaN unless status is
    RAY_OK); the projection of the slowness itself is the receiver's travel time, bit for bit."""
    values: np.ndarray    # float32[S, R]
    status: np.ndarray    # int32[S, R]
    length: np.ndarray    # int32[S, R]
    stats: SweepStats


@dataclass
class Backprojection:
    """G^T*w (SweepContext.ray_backproject): grad[nx, ny, nz] = sum over the OK rays of w times the half edge length
    of every ray edge touching the node, accumulated exactly in integer quanta of 2^quantum_exp and rounded once."""
    grad: np.ndarray      # float32[nx, ny, nz]
    quantum_exp: int
    status: np.ndarray    # int32[S, R]
    stats: SweepStats


@dataclass
class MisfitGradient:
    """misfit_gradient: misfit = 1/2 sum residual^2 (float64) over the OK rays with a pick; residual[s, r] =
    float32(tt_receiver - observed), NaN where the ray is not OK or has no pick; gradient = G^T*residual over those
    rays (ray_backproject, quantum 2^quantum_exp)."""
    misfit: float
    gradient: np.ndarray  # float32[nx, ny, nz]
    residual: np.ndarray  # float32[S, R]
    status: np.ndarray    # int32[S, R]
    quantum_exp: int


@dataclass
class LinearizedUpdate:
    """linearized_update: delta (float32[nx, ny, nz]) is the damped least-squares slowness perturbation of one
    linearised step (LSQR over the frozen rays); residual[s, r] = float32(observed - t), NaN where the ray is not OK
    or has no pick; misfit = 1/2 sum residual^2 (float64) before the step; istop, iterations and residual_norm
    (||r - G delta||, LSQR's r1norm) as scipy.sparse.linalg.lsqr reports them."""
    delta: np.ndarray     # float32[nx, ny, nz]
    residual: np.ndarray  # float32[S, R]
    status: np.ndarray    # int32[S, R]
    misfit: float
    istop: int
    iterations: int
    residual_norm: float


@dataclass
class LsqrSolution:
    """RaySet.lsqr: x (float64[nx, ny, nz]) minimises ||G_rows x - b||^2 + smooth^2 ||D x||^2 + damp^2 ||x||^2; istop,
    itn and the six norms mean what scipy.sparse.linalg.lsqr's return tuple means."""
    x: np.ndarray         # float64[nx, ny, nz]
    istop: int
    itn: int
    r1norm: float
    r2norm: float
    anorm: float
    acond: float
    arnorm: float
    xnorm: float
    stats: SweepStats


@dataclass
class Locations:
    """Events located by grid search (SweepContext.locate_events): for event e, node[e] (caller axes) minimises the
    float64 least-squares misfit of its picks with the origin time eliminated, ties to the smallest FLOATBOX index;
    misfit[e] is that minimum rounded to float32 and origin_time[e] the origin time there.  status[e] is LOC_OK,
    LOC_NO_PICKS (npicks[e] = 0) or LOC_UNREACHED (every node has an infinite time at a picked station); then node is
    (-1, -1, -1), misfit +inf and origin_time NaN."""
    node: np.ndarray         # int32[E, 3]
    misfit: np.ndarray       # float32[E]
    origin_time: np.ndarray  # float64[E]
    npicks: np.ndarray       # int32[E]
    status: np.ndarray       # int32[E]
    stats: SweepStats


@dataclass
class MisfitRegions:
    """The region R_e = {n : misfit_e(n) <= level_e} of every event, summarised exactly on the device
    (SweepContext.misfit_regions, include/sweeptt.h sweeptt_misfit_regions).  count[e] = |R_e|; lo[e] / hi[e] the
    inclusive caller-axis bounding box (-1 when empty); moments[e] = S0 S1 S2 S00 S11 S22 S01 S02 S12, the integer sums
    of c_a and c_a*c_b over the node coordinates c in R_e; origin_min / origin_max the extremes of the origin time over
    R_e (NaN when empty); npicks and status as in Locations."""
    count: np.ndarray        # int64[E]
    lo: np.ndarray           # int32[E, 3]
    hi: np.ndarray           # int32[E, 3]
    moments: np.ndarray      # int64[E, 9]
    origin_min: np.ndarray   # float64[E]
    origin_max: np.ndarray   # float64[E]
    npicks: np.ndarray       # int32[E]
    status: np.ndarray       # int32[E]
    stats: SweepStats

    def mean(self) -> np.ndarray:
        """float64 [E, 3]: the mean node coordinate of each region, each value the exact quotient rounded once; NaN
        where the region is empty."""
        from fractions import Fraction
        out = np.full((len(self.count), 3), np.nan)
        for e, n in enumerate(self.count.tolist()):
            if n:
                for a in range(3):
                    out[e, a] = float(Fraction(int(self.moments[e, a]), n))
        return out

    def covariance(self) -> np.ndarray:
        """float64 [E, 3, 3]: the population covariance of each region's node coordinates (node units),
        (n*S_ab - S_a*S_b) / n^2 computed exactly and rounded once; NaN where the region is empty."""
        from fractions import Fraction
        out = np.full((len(self.count), 3, 3), np.nan)
        second = {(0, 0): 3, (1, 1): 4, (2, 2): 5, (0, 1): 6, (0, 2): 7, (1, 2): 8}
        for e, n in enumerate(self.count.tolist()):
            if n:
                m = [int(x) for x in self.moments[e]]
                for (a, b), i in second.items():
                    out[e, a, b] = out[e, b, a] = float(Fraction(n * m[i] - m[a] * m[b], n * n))
        return out


class SweepContext:
    """Device-resident context: padded slowness box + pool of travel-time boxes on one GPU."""

    def __init__(self, *, device: int | None = None, kernel: int | None = None, loop: int | None = None,
                 max_rounds: int | None = None, star_used: int | None = None, profile_kernels: int | None = None,
                 rounds_per_poll: int | None = None, verbose: int | None = None):
        self._lib = load_library()
        o = _opts(device=device, kernel=kernel, loop=loop, max_rounds=max_rounds, star_used=star_used,
                  profile_kernels=profile_kernels, rounds_per_poll=rounds_per_poll, verbose=verbose)
        self._h = self._lib.sweeptt_create(C.byref(o))
        if not self._h:
            raise SweepError(f"sweeptt_create: {self._lib.sweeptt_last_error().decode()}")
        self.dims = None
        self.nsrc = 0
        self._sets = weakref.WeakSet()

    def close(self):
        """Closes every ray set frozen from this context that is still open, then the context."""
        if getattr(self, "_h", None):
            for rs in list(self._sets):
                rs.close()
            self._lib.sweeptt_destroy(self._h)
            self._h = None

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def set_stream(self, cuda_stream: int):
        _check(self._lib.sweeptt_set_stream(self._h, C.c_void_p(cuda_stream)), "sweeptt_set_stream")

    def set_model(self, slowness):
        v = np.ascontiguousarray(slowness, dtype=np.float32)
        _check(self._lib.sweeptt_set_model(self._h, v.ctypes.data, *v.shape), "sweeptt_set_model")
        self.dims = v.shape  # (a refused model leaves the previous one, and its dimensions)

    def set_star(self, star, delta: float = 10.0):
        fs = _as_star(star, delta)
        _check(self._lib.sweeptt_set_star(self._h, fs, len(fs)), "sweeptt_set_star")

    def set_sources(self, starts):
        st = _make_starts(starts)
        _check(self._lib.sweeptt_set_sources(self._h, st, len(st)), "sweeptt_set_sources")
        self.nsrc = len(st)

    def run(self) -> SweepStats:
        s = _Stats()
        _check(self._lib.sweeptt_run(self._h, C.byref(s)), "sweeptt_run")
        return SweepStats._from(s)

    def reset(self):
        _check(self._lib.sweeptt_reset(self._h), "sweeptt_reset")

    def step(self, rounds: int = 1):
        s = _Stats()
        ch = C.c_int(0)
        _check(self._lib.sweeptt_step(self._h, rounds, C.byref(ch), C.byref(s)), "sweeptt_step")
        return bool(ch.value), SweepStats._from(s)

    def get_tt(self, source: int, out=None):
        if out is None:
            out = np.empty(self.dims, np.float32)
        _check(self._lib.sweeptt_get_tt(self._h, source, out.ctypes.data), "sweeptt_get_tt")
        return out

    def put_tt(self, source: int, tt):
        t = np.ascontiguousarray(tt, dtype=np.float32)
        _check(self._lib.sweeptt_put_tt(self._h, source, t.ctypes.data), "sweeptt_put_tt")

    def count_violations(self, source: int) -> int:
        n = C.c_longlong(0)
        _check(self._lib.sweeptt_count_violations(self._h, source, C.byref(n)), "sweeptt_count_violations")
        return n.value

    def _source_range(self, sources, who):
        if sources is None:
            return 0, self.nsrc
        if isinstance(sources, range):
            if sources.step != 1:
                raise SweepError(f"{who}: sources must be a contiguous range")
            return sources.start, len(sources)
        begin, count = (int(x) for x in sources)
        return begin, count

    def _ray_calls(self, max_nodes, call):
        """The max_nodes policy of the ray calls: call(cap) -> (result, status), repeated with twice the capacity
        (from nx+ny+nz) while a ray is RAY_TRUNCATED, unless max_nodes is given."""
        grow = max_nodes is None
        cap = int(max_nodes) if max_nodes is not None else (sum(self.dims) if self.dims else 1)
        while True:
            out, status = call(cap)
            if not (grow and (status == RAY_TRUNCATED).any()):
                return out
            cap *= 2

    def trace_rays(self, receivers, sources=None, max_nodes: int | None = None) -> Rays:
        """Shortest-path rays from every receiver (R,3) back to the start of every source in `sources` (a range or a
        (begin, count) pair; default: all), read off the converged fields on the device (include/sweeptt.h,
        sweeptt_trace_rays).  The default max_nodes is nx+ny+nz; when a ray is longer the call is repeated with
        twice the capacity until none is truncated.  An explicit max_nodes is kept, and longer rays come back
        RAY_TRUNCATED."""
        begin, count = self._source_range(sources, "trace_rays")
        rec = _make_starts(receivers)
        nrec = len(rec)

        def call(cap):
            tt = np.empty((count, nrec), np.float32)
            status = np.empty((count, nrec), np.int32)
            length = np.empty((count, nrec), np.int32)
            nodes = np.full((count, nrec, cap, 3), -1, np.int32)
            s = _Stats()
            _check(self._lib.sweeptt_trace_rays(self._h, begin, count, rec, nrec, cap, nodes.ctypes.data,
                                                length.ctypes.data, status.ctypes.data, tt.ctypes.data, C.byref(s)),
                   "sweeptt_trace_rays")
            return Rays(tt, status, length, nodes, SweepStats._from(s)), status

        return self._ray_calls(max_nodes, call)

    def ray_project(self, perturbation, receivers, sources=None, max_nodes: int | None = None) -> RayProjection:
        """G*d: the perturbation (nx, ny, nz) summed along the ray of every (source, receiver) pair, on the device
        (include/sweeptt.h, sweeptt_ray_project).  Sources and max_nodes as in trace_rays."""
        begin, count = self._source_range(sources, "ray_project")
        d = np.ascontiguousarray(perturbation, dtype=np.float32)
        if self.dims is None or d.shape != tuple(self.dims):
            raise SweepError(f"ray_project: perturbation of shape {d.shape}, the model is {self.dims}")
        rec = _make_starts(receivers)
        nrec = len(rec)

        def call(cap):
            values = np.empty((count, nrec), np.float32)
            status = np.empty((count, nrec), np.int32)
            length = np.empty((count, nrec), np.int32)
            s = _Stats()
            _check(self._lib.sweeptt_ray_project(self._h, begin, count, rec, nrec, cap, d.ctypes.data,
                                                 values.ctypes.data, status.ctypes.data, length.ctypes.data,
                                                 C.byref(s)), "sweeptt_ray_project")
            return RayProjection(values, status, length, SweepStats._from(s)), status

        return self._ray_calls(max_nodes, call)

    def ray_backproject(self, weights, receivers, sources=None, max_nodes: int | None = None) -> Backprojection:
        """G^T*w: the weights [S, R] (finite; usually travel-time residuals) back-projected onto the grid along the
        rays, exactly and deterministically (include/sweeptt.h, sweeptt_ray_backproject).  w = 1 gives the ray
        coverage.  Sources and max_nodes as in trace_rays."""
        begin, count = self._source_range(sources, "ray_backproject")
        rec = _make_starts(receivers)
        nrec = len(rec)
        w = np.ascontiguousarray(weights, dtype=np.float32)
        if w.shape != (count, nrec):
            raise SweepError(f"ray_backproject: weights of shape {w.shape}, expected {(count, nrec)}")

        def call(cap):
            grad = np.empty(self.dims, np.float32)
            status = np.empty((count, nrec), np.int32)
            e = C.c_int(0)
            s = _Stats()
            _check(self._lib.sweeptt_ray_backproject(self._h, begin, count, rec, nrec, cap, w.ctypes.data,
                                                     grad.ctypes.data, C.byref(e), status.ctypes.data, C.byref(s)),
                   "sweeptt_ray_backproject")
            return Backprojection(grad, e.value, status, SweepStats._from(s)), status

        return self._ray_calls(max_nodes, call)

    def freeze_rays(self, receivers, sources=None, max_nodes: int | None = None) -> "RaySet":
        """Traces the rays of trace_rays once and keeps them on the device as a RaySet (include/sweeptt.h,
        sweeptt_rayset_freeze), whose project / backproject equal ray_project / ray_backproject of this context as it
        is now, bit for bit, however the context changes later.  Sources and max_nodes as in trace_rays: with the
        default the freeze is repeated at twice the capacity while a ray is RAY_TRUNCATED."""
        begin, count = self._source_range(sources, "freeze_rays")
        rec = _make_starts(receivers)
        nrec = len(rec)

        def call(cap):
            s = _Stats()
            h = self._lib.sweeptt_rayset_freeze(self._h, begin, count, rec, nrec, cap, C.byref(s))
            if not h:
                raise SweepError(f"sweeptt_rayset_freeze: {self._lib.sweeptt_last_error().decode()}")
            rs = RaySet(self, h, (count, nrec), tuple(self.dims), SweepStats._from(s))
            if grow and (rs.status == RAY_TRUNCATED).any():
                rs.close()
            return rs, rs.status

        grow = max_nodes is None
        rs = self._ray_calls(max_nodes, call)
        self._sets.add(rs)
        return rs

    def locate_events(self, picks, sources=None) -> Locations:
        """Locates every event of picks [E, S] (float32, NaN = no pick) by grid search over the fields of the sources
        in `sources` (the stations; a range or a (begin, count) pair; default: all), on the device (include/sweeptt.h,
        sweeptt_locate_events).  The misfit is computed in float64 exactly as the header states it."""
        begin, count = self._source_range(sources, "locate_events")
        p = np.ascontiguousarray(picks, dtype=np.float32)
        if p.ndim != 2 or p.shape[1] != count:
            raise SweepError(f"locate_events: picks of shape {p.shape}, expected (events, {count})")
        nev = p.shape[0]
        node = np.empty((nev, 3), np.int32)
        misfit = np.empty(nev, np.float32)
        origin = np.empty(nev, np.float64)
        npicks = np.empty(nev, np.int32)
        status = np.empty(nev, np.int32)
        s = _Stats()
        _check(self._lib.sweeptt_locate_events(self._h, begin, count, p.ctypes.data, nev, node.ctypes.data,
                                               misfit.ctypes.data, origin.ctypes.data, npicks.ctypes.data,
                                               status.ctypes.data, C.byref(s)), "sweeptt_locate_events")
        return Locations(node, misfit, origin, npicks, status, SweepStats._from(s))

    def misfit_regions(self, picks, levels, sources=None) -> MisfitRegions:
        """The nodes of every event of picks [E, S] whose misfit is at most levels[e] (float32 [E]; finite and >= 0, or
        NaN for no region), summarised exactly on the device: count, bounding box, integer moments and origin-time range
        (include/sweeptt.h, sweeptt_misfit_regions).  The region is exactly misfit_box(picks[e]) <= levels[e]; an event
        without a pick has an empty one.  Sources as in locate_events."""
        begin, count = self._source_range(sources, "misfit_regions")
        p = np.ascontiguousarray(picks, dtype=np.float32)
        if p.ndim != 2 or p.shape[1] != count:
            raise SweepError(f"misfit_regions: picks of shape {p.shape}, expected (events, {count})")
        nev = p.shape[0]
        lv = np.ascontiguousarray(levels, dtype=np.float32)
        if lv.shape != (nev,):
            raise SweepError(f"misfit_regions: levels of shape {lv.shape}, expected ({nev},)")
        n = np.empty(nev, np.int64)
        bbox = np.empty((nev, 6), np.int32)
        moments = np.empty((nev, 9), np.int64)
        origin = np.empty((nev, 2), np.float64)
        status = np.empty(nev, np.int32)
        s = _Stats()
        _check(self._lib.sweeptt_misfit_regions(self._h, begin, count, p.ctypes.data, nev, lv.ctypes.data, n.ctypes.data,
                                                bbox.ctypes.data, moments.ctypes.data, origin.ctypes.data,
                                                status.ctypes.data, C.byref(s)), "sweeptt_misfit_regions")
        npicks = (~np.isnan(p)).sum(1).astype(np.int32)
        return MisfitRegions(n, bbox[:, :3].copy(), bbox[:, 3:].copy(), moments, origin[:, 0].copy(),
                             origin[:, 1].copy(), npicks, status, SweepStats._from(s))

    def misfit_box(self, picks, sources=None) -> np.ndarray:
        """The misfit of one event (picks [S], NaN = no pick) at every node: float32[nx, ny, nz], +inf where a picked
        station's time is infinite (include/sweeptt.h, sweeptt_misfit_box).  locate_events returns its argmin."""
        begin, count = self._source_range(sources, "misfit_box")
        p = np.ascontiguousarray(picks, dtype=np.float32)
        if p.shape != (count,):
            raise SweepError(f"misfit_box: picks of shape {p.shape}, expected ({count},)")
        if self.dims is None:
            raise SweepError("misfit_box: the context needs a model first")
        out = np.empty(self.dims, np.float32)
        s = _Stats()
        _check(self._lib.sweeptt_misfit_box(self._h, begin, count, p.ctypes.data, out.ctypes.data, C.byref(s)),
               "sweeptt_misfit_box")
        return out

    @property
    def relaxations_per_round(self) -> int:
        return self._lib.sweeptt_relaxations_per_round(self._h)

    @property
    def tiles_per_source(self) -> int:
        return self._lib.sweeptt_tiles_per_source(self._h)

    @property
    def pool_bytes(self) -> int:
        return self._lib.sweeptt_pool_bytes(self._h)

    def model_stats(self):
        """Test hook: (vmin, vmax, vpos) the context keeps of its model (include/sweeptt.h)."""
        out = np.zeros(3, np.float32)
        _check(self._lib.sweeptt_debug_model_stats(self._h, out[0:].ctypes.data, out[1:].ctypes.data,
                                                   out[2:].ctypes.data), "sweeptt_debug_model_stats")
        return tuple(out)


class RaySet:
    """Rays of sources [S] x receivers [R] traced once and kept on the device (SweepContext.freeze_rays): G*d and G^T*w
    from the stored rays, bit for bit what ray_project / ray_backproject gave at the freeze.  A snapshot: later changes
    of the context (model, star, fields) leave it unchanged.  Close it (or its context) to release nbytes of device
    memory; a closed set raises."""

    def __init__(self, ctx: SweepContext, handle, shape, dims, stats: SweepStats):
        self._lib = ctx._lib
        self._ctx = ctx              # the context outlives its sets
        self._h = handle
        self.shape = shape           # (S, R)
        self.dims = dims             # (nx, ny, nz) of the model at the freeze
        self.stats = stats           # of the freeze
        self.length = np.empty(shape, np.int32)
        self.status = np.empty(shape, np.int32)
        self.tt = np.empty(shape, np.float32)
        _check(self._lib.sweeptt_rayset_table(self._h, self.length.ctypes.data, self.status.ctypes.data,
                                              self.tt.ctypes.data), "sweeptt_rayset_table")

    def _handle(self):
        if not self._h:
            raise SweepError("ray set is closed")
        return self._h

    def close(self):
        if getattr(self, "_h", None):
            self._lib.sweeptt_rayset_destroy(self._h)
            self._h = None

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    @property
    def nbytes(self) -> int:
        """Device memory the set holds (include/sweeptt.h, sweeptt_rayset_bytes)."""
        return self._lib.sweeptt_rayset_bytes(self._handle())

    def project(self, perturbation) -> RayProjection:
        """G*d over every ray of the set (values NaN unless status is RAY_OK)."""
        d = np.ascontiguousarray(perturbation, dtype=np.float32)
        if d.shape != self.dims:
            raise SweepError(f"RaySet.project: perturbation of shape {d.shape}, the rays are on {self.dims}")
        values = np.empty(self.shape, np.float32)
        s = _Stats()
        _check(self._lib.sweeptt_rayset_project(self._handle(), d.ctypes.data, values.ctypes.data, C.byref(s)),
               "sweeptt_rayset_project")
        return RayProjection(values, self.status, self.length, SweepStats._from(s))

    def backproject(self, weights) -> Backprojection:
        """G^T*w over every ray of the set; weights [S, R] finite (only the OK rays contribute)."""
        w = np.ascontiguousarray(weights, dtype=np.float32)
        if w.shape != self.shape:
            raise SweepError(f"RaySet.backproject: weights of shape {w.shape}, expected {self.shape}")
        grad = np.empty(self.dims, np.float32)
        e = C.c_int(0)
        s = _Stats()
        _check(self._lib.sweeptt_rayset_backproject(self._handle(), w.ctypes.data, grad.ctypes.data, C.byref(e),
                                                    C.byref(s)), "sweeptt_rayset_backproject")
        return Backprojection(grad, e.value, self.status, SweepStats._from(s))

    def paths(self):
        """(offsets int64[S*R+1], nodes int32[offsets[-1], 3]): ray q = s*R + r has the nodes
        nodes[offsets[q]:offsets[q+1]] (caller axes, receiver first); rays that are not OK have none."""
        h = self._handle()
        offsets = np.empty(self.status.size + 1, np.int64)
        _check(self._lib.sweeptt_rayset_paths(h, offsets.ctypes.data, None), "sweeptt_rayset_paths")
        nodes = np.empty((int(offsets[-1]), 3), np.int32)
        _check(self._lib.sweeptt_rayset_paths(h, None, nodes.ctypes.data), "sweeptt_rayset_paths")
        return offsets, nodes

    def as_linear_operator(self, rows=None):
        """G as a scipy.sparse.linalg.LinearOperator (float64) over the rays selected by rows (bool [S, R]; default:
        the OK rays) and every node of the box (raveled FLOATBOX order).  The conversions are part of the definition:
          matvec(x)  = float64(project(float32(x)).values[rows])
          rmatvec(y) = float64(backproject(W).grad).ravel(), W = float32(y) scattered into [S, R], 0 outside rows.
        Both run on the device; only the vectors cross PCIe."""
        from scipy.sparse.linalg import LinearOperator
        rows = self.status == RAY_OK if rows is None else np.asarray(rows, bool)
        if rows.shape != self.shape:
            raise SweepError(f"RaySet.as_linear_operator: rows of shape {rows.shape}, expected {self.shape}")
        if not (self.status[rows] == RAY_OK).all():
            raise SweepError("RaySet.as_linear_operator: rows selects a ray that is not OK")
        n = int(np.prod(self.dims))

        def matvec(x):
            d = np.asarray(x, np.float32).reshape(self.dims)
            return self.project(d).values[rows].astype(np.float64)

        def rmatvec(y):
            w = np.zeros(self.shape, np.float32)
            w[rows] = np.asarray(y, np.float32).ravel()
            return self.backproject(w).grad.astype(np.float64).ravel()

        return LinearOperator((int(rows.sum()), n), matvec=matvec, rmatvec=rmatvec, dtype=np.float64)

    def lsqr(self, b, rows=None, *, damp: float = 0.0, smooth: float = 0.0, atol: float = 1e-6, btol: float = 1e-6,
             conlim: float = 1e8, iter_lim: int | None = None) -> LsqrSolution:
        """scipy.sparse.linalg.lsqr on the device (include/sweeptt.h, sweeptt_rayset_lsqr): minimises
        ||A x - [b; 0]||^2 + damp^2 ||x||^2 with A = [G_rows; smooth D], G_rows = as_linear_operator(rows) (rows: bool
        [S, R], default the OK rays; b: float64 over the selected rays in q order) and D the first difference along
        every axis.  Only b goes to the device and only x and a few scalars per iteration come back.  iter_lim None is
        scipy's 2 nx ny nz."""
        rows = self.status == RAY_OK if rows is None else np.asarray(rows, bool)
        if rows.shape != self.shape:
            raise SweepError(f"RaySet.lsqr: rows of shape {rows.shape}, expected {self.shape}")
        bb = np.ascontiguousarray(b, dtype=np.float64).ravel()
        if bb.size != int(rows.sum()):
            raise SweepError(f"RaySet.lsqr: b has {bb.size} values, rows selects {int(rows.sum())} rays")
        sel = np.ascontiguousarray(rows, dtype=np.uint8)
        n = int(np.prod(self.dims))
        opts = _LsqrOpts(C.sizeof(_LsqrOpts), damp, smooth, atol, btol, conlim, 2 * n if iter_lim is None else iter_lim)
        info = _LsqrInfo(C.sizeof(_LsqrInfo))
        x = np.empty(self.dims, np.float64)
        s = _Stats()
        _check(self._lib.sweeptt_rayset_lsqr(self._handle(), sel.ctypes.data, bb.ctypes.data, C.byref(opts),
                                             x.ctypes.data, C.byref(info), C.byref(s)), "sweeptt_rayset_lsqr")
        return LsqrSolution(x, info.istop, info.itn, info.r1norm, info.r2norm, info.anorm, info.acond, info.arnorm,
                            info.xnorm, SweepStats._from(s))


def trace_rays(slowness, star, starts, receivers, *, delta: float = 10.0, max_nodes: int | None = None,
               device: int | None = None, kernel: int | None = None, star_used: int | None = None) -> Rays:
    """One-shot: solve every start on one device, then trace rays from every receiver back to each start
    (SweepContext.trace_rays).  Only the rays and receiver times leave the device, never the fields."""
    with SweepContext(device=device, kernel=kernel, star_used=star_used) as ctx:
        ctx.set_model(slowness)
        ctx.set_star(star, delta)
        ctx.set_sources(starts)
        ctx.run()
        return ctx.trace_rays(receivers, max_nodes=max_nodes)


def misfit_gradient(slowness, star, starts, receivers, observed, *, delta: float = 10.0, device: int | None = None,
                    kernel: int | None = None, star_used: int | None = None) -> MisfitGradient:
    """One-shot gradient of the ray-linearised travel-time misfit 1/2 sum (t - observed)^2 with respect to slowness.

    Solves every start, reads the receiver times (trace_rays with max_nodes=1: one step per ray), forms
    residual = float32(t - observed) (a NaN in observed [S, R] means no pick: weight 0) and back-projects the residuals
    of the OK rays (SweepContext.ray_backproject).  The misfit is summed in float64 over the OK rays with a pick; every
    other residual is NaN, and the gradient equals ray_backproject of the residuals with those NaN set to 0.

    The gradient is that of the misfit with the rays held fixed.  The discrete travel time is a minimum over paths of
    sums linear in the slowness, so it is concave: the row of G of a ray is a supergradient of that ray's travel time
    (T(v + h) <= T(v) + G h up to rounding), and its exact derivative wherever the predecessor of every node on the ray
    is unique."""
    obs = np.asarray(observed, dtype=np.float32)
    with SweepContext(device=device, kernel=kernel, star_used=star_used) as ctx:
        ctx.set_model(slowness)
        ctx.set_star(star, delta)
        ctx.set_sources(starts)
        ctx.run()
        rec = _make_starts(receivers)
        if obs.shape != (ctx.nsrc, len(rec)):
            raise SweepError(f"misfit_gradient: observed of shape {obs.shape}, expected {(ctx.nsrc, len(rec))}")
        t = ctx.trace_rays(receivers, max_nodes=1).tt
        with np.errstate(invalid="ignore", over="ignore"):
            residual = (t - obs).astype(np.float32)
        use = np.isfinite(residual)   # a pick, and a reached receiver
        while True:
            bp = ctx.ray_backproject(np.where(use, residual, np.float32(0)), receivers)
            ok = use & (bp.status == RAY_OK)
            if (ok == use).all():
                break
            use = ok   # a ray with a weight turned out not OK: drop it, so the quantum depends on the used rays only
    residual = np.where(use, residual, np.float32(np.nan)).astype(np.float32)
    misfit = 0.5 * float(np.sum(residual[use].astype(np.float64) ** 2))
    return MisfitGradient(misfit, bp.grad, residual, bp.status, bp.quantum_exp)


def linearized_update(slowness, star, starts, receivers, observed, *, damp: float, iter_lim: int,
                      atol: float = 1e-6, btol: float = 1e-6, delta: float = 10.0, device: int | None = None,
                      kernel: int | None = None, star_used: int | None = None) -> LinearizedUpdate:
    """One damped linearised inversion step: the slowness perturbation that minimises ||G d - r||^2 + damp^2 ||d||^2
    with the rays held fixed.  The companion of misfit_gradient, with its pick rule.

    Solves every start, freezes the rays (SweepContext.freeze_rays), forms r = float32(observed - t) over the OK rays
    with a pick (a NaN in observed [S, R] means no pick) and runs scipy.sparse.linalg.lsqr(G, r, damp, atol, btol,
    iter_lim) on RaySet.as_linear_operator of those rays, every operator applied on the device from the frozen rays.
    The update is returned, not applied: clamping the slowness and re-solving are the caller's policy.

    G holds the rays fixed.  The discrete travel time is a minimum over paths of sums linear in the slowness, so it is
    concave: the row of G of a ray is a supergradient of that ray's travel time (T(v + h) <= T(v) + G h up to
    rounding), and its exact derivative wherever the predecessor of every node on the ray is unique."""
    from scipy.sparse.linalg import lsqr
    obs = np.asarray(observed, dtype=np.float32)
    with SweepContext(device=device, kernel=kernel, star_used=star_used) as ctx:
        ctx.set_model(slowness)
        ctx.set_star(star, delta)
        ctx.set_sources(starts)
        ctx.run()
        nrec = len(_make_starts(receivers))
        if obs.shape != (ctx.nsrc, nrec):
            raise SweepError(f"linearized_update: observed of shape {obs.shape}, expected {(ctx.nsrc, nrec)}")
        with ctx.freeze_rays(receivers) as rs:
            with np.errstate(invalid="ignore", over="ignore"):
                residual = (obs - rs.tt).astype(np.float32)
            use = np.isfinite(residual) & (rs.status == RAY_OK)
            residual = np.where(use, residual, np.float32(np.nan)).astype(np.float32)
            out = lsqr(rs.as_linear_operator(use), residual[use].astype(np.float64), damp=damp, atol=atol, btol=btol,
                       iter_lim=iter_lim)
            status = rs.status
    misfit = 0.5 * float(np.sum(residual[use].astype(np.float64) ** 2))
    return LinearizedUpdate(out[0].astype(np.float32).reshape(np.shape(slowness)), residual, status, misfit,
                            int(out[1]), int(out[2]), float(out[3]))


def locate_events(slowness, star, stations, picks, *, delta: float = 10.0, device: int | None = None,
                  kernel: int | None = None) -> Locations:
    """One-shot event location: solve one field per station (stations (S, 3) as start points; by reciprocity the
    field of station s holds the time from every node to s), then locate every event of picks [E, S]
    (SweepContext.locate_events).  Only the locations leave the device, never the fields."""
    with SweepContext(device=device, kernel=kernel) as ctx:
        ctx.set_model(slowness)
        ctx.set_star(star, delta)
        ctx.set_sources(stations)
        ctx.run()
        return ctx.locate_events(picks)


def uncertainty_levels(locations: Locations, sigma, confidence: float = 0.95) -> np.ndarray:
    """The levels of location_uncertainty: float32(float64(misfit) + sigma^2 * chi2.ppf(confidence, 3)) for the
    events located OK, NaN for the others and where the best misfit overflowed to +inf; a sum beyond float32 becomes
    its largest finite value (every node with a finite misfit is then inside)."""
    from scipy.stats import chi2
    misfit = np.asarray(locations.misfit, np.float32)
    sig = np.broadcast_to(np.asarray(sigma, np.float64), misfit.shape)
    if not (np.isfinite(sig).all() and (sig > 0).all()):
        raise SweepError("location_uncertainty: sigma must be finite and > 0")
    if not 0.0 < confidence < 1.0:
        raise SweepError(f"location_uncertainty: confidence {confidence} is not in (0, 1)")
    ok = (np.asarray(locations.status) == LOC_OK) & np.isfinite(misfit)
    with np.errstate(over="ignore"):
        lv = (misfit.astype(np.float64) + sig * sig * float(chi2.ppf(confidence, 3))).astype(np.float32)
    lv = np.where(np.isinf(lv), np.finfo(np.float32).max, lv)
    return np.where(ok, lv, np.float32(np.nan)).astype(np.float32)


def location_uncertainty(slowness, star, stations, picks, *, sigma, confidence: float = 0.95, delta: float = 10.0,
                         device: int | None = None, kernel: int | None = None):
    """One-shot location with uncertainty: on one context, solve one field per station, locate every event of picks
    [E, S] (SweepContext.locate_events), then summarise each event's confidence region (SweepContext.misfit_regions)
    at the level misfit_best + sigma^2 * chi2.ppf(confidence, 3) (uncertainty_levels).  Returns (Locations,
    MisfitRegions).

    The statistical assumption: the picks are the fields' times at the true node plus a common origin time plus
    independent Gaussian errors of standard deviation sigma (a scalar or one value per event, finite and > 0, in the
    fields' units).  Then the misfit, with the origin time profiled out, exceeds its minimum by sigma^2 times a
    chi-square variable of 3 degrees of freedom (the three coordinates) at the true node, in the linearised limit, and
    the region is the usual delta-chi-square confidence region at that confidence.  The discretisation of the grid is
    not part of it: the region is a set of nodes, and a region of one node says the grid is too coarse to resolve
    the uncertainty, not that there is none."""
    with SweepContext(device=device, kernel=kernel) as ctx:
        ctx.set_model(slowness)
        ctx.set_star(star, delta)
        ctx.set_sources(stations)
        ctx.run()
        loc = ctx.locate_events(picks)
        return loc, ctx.misfit_regions(picks, uncertainty_levels(loc, sigma, confidence))


# ---- file formats -------------------------------------------------------------------------

def _take_floats(ptr, dims):
    n = int(dims[0]) * int(dims[1]) * int(dims[2])
    arr = np.ctypeslib.as_array(ptr, shape=(n,)).reshape(tuple(int(d) for d in dims)).copy()
    load_library().sweeptt_free(ptr)
    return arr


def vbox_load(path):
    lib = load_library()
    p = C.POINTER(C.c_float)()
    o, d = (C.c_int * 3)(), (C.c_int * 3)()
    _check(lib.sweeptt_vbox_load(os.fsencode(path), C.byref(p), o, d), "sweeptt_vbox_load")
    return _take_floats(p, d), tuple(o), tuple(d)


def vbox_store(path, slowness, origin=(0, 0, 0)):
    v = np.ascontiguousarray(slowness, dtype=np.float32)
    o, d = (C.c_int * 3)(*origin), (C.c_int * 3)(*v.shape)
    _check(load_library().sweeptt_vbox_store(os.fsencode(path), v.ctypes.data, o, d), "sweeptt_vbox_store")


def vbox_load_subset(path, sub_origin, sub_dims):
    p = C.POINTER(C.c_float)()
    o, d = (C.c_int * 3)(*sub_origin), (C.c_int * 3)(*sub_dims)
    _check(load_library().sweeptt_vbox_load_subset(os.fsencode(path), o, d, C.byref(p)), "sweeptt_vbox_load_subset")
    return _take_floats(p, d)


def text_load(path):
    p = C.POINTER(C.c_float)()
    o, d = (C.c_int * 3)(), (C.c_int * 3)()
    _check(load_library().sweeptt_text_load(os.fsencode(path), C.byref(p), o, d), "sweeptt_text_load")
    return _take_floats(p, d), tuple(o), tuple(d)


def star_load(path, delta: float = 10.0):
    lib = load_library()
    p = C.POINTER(FS)()
    n = C.c_int(0)
    _check(lib.sweeptt_star_load(os.fsencode(path), C.c_float(delta), C.byref(p), C.byref(n)), "sweeptt_star_load")
    off = np.array([(p[l].i, p[l].j, p[l].k) for l in range(n.value)], np.int32)
    d = np.array([p[l].d for l in range(n.value)], np.float32)
    lib.sweeptt_free(p)
    return off, d


def starts_load(path):
    lib = load_library()
    p = C.POINTER(START)()
    n = C.c_int(0)
    _check(lib.sweeptt_starts_load(os.fsencode(path), C.byref(p), C.byref(n)), "sweeptt_starts_load")
    st = np.array([(p[s].i, p[s].j, p[s].k) for s in range(n.value)], np.int32)
    lib.sweeptt_free(p)
    return st


def write_output_tt(path, tt):
    t = np.ascontiguousarray(tt, dtype=np.float32)
    ns, nx, ny, nz = t.shape
    ptrs = (C.c_void_p * ns)(*[t[s].ctypes.data for s in range(ns)])
    _check(load_library().sweeptt_write_output_tt(os.fsencode(path), ptrs, ns, nx, ny, nz), "sweeptt_write_output_tt")
