"""B200-native multi-start forward-star travel-time sweep (one hot path of
scrasmussen/uoparallel-seismic-project), behind a C ABI (include/sweeptt.h).

The compute lives in ``lib/libsweeptt.so`` (hand-written sm_100a CUDA, built in-tree by
``__graft_entry__.build()`` / ``csrc/Makefile``).  This package is the thin Python host
mirror used by the tests and ``bench.py``; there is no CPU fallback -- every compute call
raises ``SweepError`` when the extension or a CUDA device is missing.
"""
from .api import (  # noqa: F401
    FS,
    Backprojection,
    LOC_NO_PICKS,
    LOC_OK,
    LOC_UNREACHED,
    LinearizedUpdate,
    Locations,
    LsqrSolution,
    MisfitGradient,
    MisfitRegions,
    RayProjection,
    RaySet,
    Rays,
    START,
    SweepContext,
    SweepError,
    SweepStats,
    build_pull_star,
    device_count,
    lib_path,
    load_library,
    linearized_update,
    locate_events,
    location_uncertainty,
    make_star,
    solve,
    solve_slabs,
    solve_slabs_vbox,
    star_load,
    starts_load,
    text_load,
    misfit_gradient,
    trace_rays,
    uncertainty_levels,
    vbox_load,
    vbox_load_subset,
    vbox_store,
    write_output_tt,
)
from . import workloads  # noqa: F401
