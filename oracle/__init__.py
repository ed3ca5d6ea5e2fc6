"""Parity oracle (TEST INFRASTRUCTURE ONLY -- see oracle/sweep_oracle.c header).

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference leg may
import this package.  `restatement()` is our C restatement; `reference()` is the reference's
own serial_new program compiled into oracle/_ref from the checkout of the original project named by
$SWEEPTT_REFERENCE (None when absent).
"""
from __future__ import annotations

import ctypes as C
import pathlib
import subprocess

import numpy as np

_HERE = pathlib.Path(__file__).resolve().parent
_LIB = None
_REF = None


def build(quiet=True):
    subprocess.run(["make", "-C", str(_HERE)], check=True,
                   stdout=subprocess.DEVNULL if quiet else None, stderr=subprocess.STDOUT if quiet else None)


def restatement() -> C.CDLL:
    global _LIB
    if _LIB is None:
        p = _HERE / "liboracle.so"
        if not p.exists():
            build()
        lib = C.CDLL(str(p))
        lib.oracle_visits_per_sweep.restype = C.c_longlong
        lib.oracle_sweep.restype = C.c_longlong
        lib.oracle_violations.restype = C.c_longlong
        lib.oracle_vbox_checksum.restype = C.c_uint32
        _LIB = lib
    return _LIB


def reference():
    """ctypes handle on the reference's own code (oracle/_ref/libref_sweep.so) or None."""
    global _REF
    if _REF is None:
        p = _HERE / "_ref" / "libref_sweep.so"
        if not p.exists():
            return None
        lib = C.CDLL(str(p))
        lib.refh_star_distance.restype = C.c_float
        lib.refh_velocity_ptr.restype = C.POINTER(C.c_float)
        _REF = lib
    return _REF


def vconvert_path():
    p = _HERE / "_ref" / "vconvert"
    return p if p.exists() else None


def _i32(a):
    return np.ascontiguousarray(a, dtype=np.int32)


def star_distances(offsets, delta=10.0):
    off = _i32(offsets).reshape(-1, 3)
    d = np.empty(len(off), np.float32)
    restatement().oracle_star_distances(off.ctypes.data_as(C.c_void_p), len(off), C.c_float(delta),
                                        d.ctypes.data_as(C.c_void_p))
    return d


def visits_per_sweep(dims, offsets, used=None):
    off = _i32(offsets).reshape(-1, 3)
    if used is None:
        used = len(off) - 1
    return restatement().oracle_visits_per_sweep(int(dims[0]), int(dims[1]), int(dims[2]),
                                                 off.ctypes.data_as(C.c_void_p), int(used))


def init_tt(dims, start):
    tt = np.full(dims, np.inf, np.float32)
    tt[tuple(int(c) for c in start)] = 0.0
    return tt


def sweep(v, tt, offsets, start, delta=10.0, used=None):
    """One in-place Gauss-Seidel sweep (restatement); returns the store count."""
    off = _i32(offsets).reshape(-1, 3)
    if used is None:
        used = len(off) - 1
    d = star_distances(off, delta)
    nx, ny, nz = v.shape
    assert v.dtype == np.float32 and tt.dtype == np.float32 and v.flags.c_contiguous and tt.flags.c_contiguous
    return restatement().oracle_sweep(v.ctypes.data_as(C.c_void_p), tt.ctypes.data_as(C.c_void_p), nx, ny, nz,
                                      off.ctypes.data_as(C.c_void_p), d.ctypes.data_as(C.c_void_p), int(used),
                                      int(start[0]), int(start[1]), int(start[2]))


def solve(v, offsets, start, delta=10.0, maxsweeps=0):
    """Sweep to convergence (restatement). Returns (tt, sweeps, stores)."""
    off = _i32(offsets).reshape(-1, 3)
    v = np.ascontiguousarray(v, np.float32)
    nx, ny, nz = v.shape
    tt = np.empty(v.shape, np.float32)
    stores = C.c_longlong(0)
    sweeps = restatement().oracle_solve(v.ctypes.data_as(C.c_void_p), tt.ctypes.data_as(C.c_void_p), nx, ny, nz,
                                        off.ctypes.data_as(C.c_void_p), len(off), C.c_float(delta), int(start[0]),
                                        int(start[1]), int(start[2]), int(maxsweeps), C.byref(stores))
    return tt, sweeps, stores.value


def violations(v, tt, offsets, start, delta=10.0, used=None):
    off = _i32(offsets).reshape(-1, 3)
    if used is None:
        used = len(off) - 1
    d = star_distances(off, delta)
    nx, ny, nz = v.shape
    v = np.ascontiguousarray(v, np.float32)
    tt = np.ascontiguousarray(tt, np.float32)
    return restatement().oracle_violations(v.ctypes.data_as(C.c_void_p), tt.ctypes.data_as(C.c_void_p), nx, ny, nz,
                                           off.ctypes.data_as(C.c_void_p), d.ctypes.data_as(C.c_void_p), int(used),
                                           int(start[0]), int(start[1]), int(start[2]))


def vbox_write(path, v, origin=(0, 0, 0)):
    v = np.ascontiguousarray(v, np.float32)
    ok = restatement().oracle_vbox_write(str(path).encode(), v.ctypes.data_as(C.c_void_p), int(origin[0]),
                                         int(origin[1]), int(origin[2]), *[int(d) for d in v.shape])
    if not ok:
        raise OSError(f"oracle_vbox_write({path}) failed")


def vbox_read(path):
    o, d = (C.c_int32 * 3)(), (C.c_int32 * 3)()
    lib = restatement()
    if not lib.oracle_vbox_read(str(path).encode(), None, o, d):
        return None
    v = np.empty(tuple(d), np.float32)
    if not lib.oracle_vbox_read(str(path).encode(), v.ctypes.data_as(C.c_void_p), o, d):
        return None
    return v, tuple(o), tuple(d)


def write_output_tt(path, tt):
    tt = np.ascontiguousarray(tt, np.float32)
    ns, nx, ny, nz = tt.shape
    ptrs = (C.c_void_p * ns)(*[tt[s].ctypes.data for s in range(ns)])
    if not restatement().oracle_write_output_tt(str(path).encode(), ptrs, ns, nx, ny, nz):
        raise OSError(f"oracle_write_output_tt({path}) failed")


# ---- the reference's own code (only where oracle/_ref was built) -----------------------------

def ref_solve(v, offsets, start, maxsweeps=0, per_sweep=None):
    """Drive the reference's unmodified sweepXYZ to convergence. Returns (tt, sweeps)."""
    lib = reference()
    if lib is None:
        raise RuntimeError("oracle/_ref not built (reference sources absent)")
    off = _i32(offsets).reshape(-1, 3)
    v = np.ascontiguousarray(v, np.float32)
    nx, ny, nz = v.shape
    assert len(off) <= lib.refh_fsmax()
    assert lib.refh_set_star(off.ctypes.data_as(C.c_void_p), len(off))
    assert lib.refh_set_velocity(v.ctypes.data_as(C.c_void_p), nx, ny, nz)
    assert lib.refh_init_source(0, int(start[0]), int(start[1]), int(start[2]))
    sweeps = 0
    tt = np.empty(v.shape, np.float32)
    while True:
        c = lib.refh_sweep_once(0, len(off))
        sweeps += 1
        if per_sweep is not None:
            lib.refh_copy_tt(0, tt.ctypes.data_as(C.c_void_p))
            per_sweep(sweeps, c, tt)
        if c == 0 or (maxsweeps and sweeps >= maxsweeps):
            break
    lib.refh_copy_tt(0, tt.ctypes.data_as(C.c_void_p))
    return tt, sweeps
