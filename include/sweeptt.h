/*
 * sweeptt.h -- C ABI of the B200-native multi-start forward-star sweep.
 *
 * This is the drop-in boundary for ONE hot path of
 * scrasmussen/uoparallel-seismic-project: "relax every grid node's travel time
 * against all offsets of a forward star until nothing changes, for every start
 * point".  Each entry point cites the reference interface it replaces
 * (paths relative to the reference checkout).
 *
 * Conventions (same polarity as the reference's loaders/allocators,
 * include/floatbox.h:118-120, include/velocityboxfiler.h:105-106):
 *   - functions returning int return NON-ZERO on success and 0 on failure;
 *     sweeptt_last_error() then holds a message (thread-local);
 *   - all boxes are FLOATBOX-ordered float32: index = (x*ny + y)*nz + z, z fastest
 *     (include/floatbox.h:127-129,160);
 *   - the caller owns every host buffer; the library owns all device memory;
 *   - there is NO CPU fallback: every compute entry point fails loudly when no
 *     CUDA device / sm_100 kernel image is available.
 *
 * Threading: a context is used by one host thread at a time.  Different contexts may be driven from different
 * threads; the forward-star tables live in per-device __constant__ memory, so contexts on ONE device whose stars
 * differ take turns (each compute call holds a lease on the device's tables for its duration; identical stars
 * share it).  Concurrent sweeptt_solve() calls for the same device serialise on that device's cached context.
 *
 * Plain C: no C++ or torch types cross this boundary.
 */
#ifndef SWEEPTT_H
#define SWEEPTT_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* serial_new/sweep-tt-multistart.c:46-49 (and cuda/cudasweep-tt-multistart.cu:58-61):
 * forward-star offset and its distance d = delta * sqrt(i*i+j*j+k*k). Layout kept.
 * A translation unit that already defines these two structs itself -- the reference's own
 * programs do -- defines SWEEPTT_NO_STRUCTS before including this header (after its own
 * definitions) and passes its arrays as they are. */
#ifndef SWEEPTT_NO_STRUCTS
struct FS {
  int i, j, k;
  float d;
};

/* serial_new/sweep-tt-multistart.c:56-58: 0-based start point. Layout kept. */
struct START {
  int i, j, k;
};
#endif

/* which relaxation kernel runs (the default is the tiled sm_100a kernel) */
enum {
  SWEEPTT_KERNEL_AUTO = 0,   /* tiled TMA kernel when the star fits its halo, else simple */
  SWEEPTT_KERNEL_SIMPLE = 1, /* one thread per node, global memory (verification path)    */
  SWEEPTT_KERNEL_TILED = 2   /* force the tiled kernel (fails if the star does not fit)   */
};

/* convergence driver */
enum {
  SWEEPTT_LOOP_AUTO = 0,
  SWEEPTT_LOOP_BATCHED = 1, /* K rounds enqueued per host poll of the device flag          */
  SWEEPTT_LOOP_GRAPH = 2    /* device-resident loop (no host poll): ONE persistent launch that builds
                               its own work lists while the activation keys fit its shared memory,
                               else a CUDA graph with a device-evaluated WHILE node              */
};

typedef struct sweeptt_opts {
  int struct_size;     /* = sizeof(sweeptt_opts); lets the struct grow compatibly           */
  int device;          /* CUDA ordinal for single-device calls; -1 = current device         */
  int num_devices;     /* sweeptt_solve only: shard sources over devices [0,num_devices);
                          0 or 1 = one device                                               */
  int kernel;          /* SWEEPTT_KERNEL_*                                                  */
  int loop;            /* SWEEPTT_LOOP_*                                                    */
  int rounds_per_poll; /* batched loop: rounds enqueued between flag reads (0 = default 8)  */
  int max_rounds;      /* safety cap on relaxation rounds (0 = none)                        */
  int star_used;       /* number of leading star entries used as sweep centres' offsets;
                          0 = starsize-1, which is what the reference passes
                          (serial_new/sweep-tt-multistart.c:160)                            */
  int verbose;         /* >0: progress lines on stderr                                      */
  int slab_axis;       /* sweeptt_solve_slabs only: 0 = x (contiguous halos), 2 = z         */
  int profile_kernels; /* !=0: bracket every relaxation launch with CUDA events (batched
                          loop) so stats.relax_kernel_ms is measured, at ~1 us per round    */
} sweeptt_opts;

typedef struct sweeptt_stats {
  int struct_size;
  int rounds;                /* relaxation rounds executed (max over sources/devices)      */
  int kernel_used;           /* SWEEPTT_KERNEL_SIMPLE or _TILED                            */
  int devices_used;
  long long kernel_launches; /* launches of OUR kernels inside the solve                   */
  long long tile_visits;     /* tiles relaxed (tiled kernel)                               */
  long long relaxations;     /* in-bounds (node, offset, source) pull evaluations executed */
  double solve_ms;           /* device time of the solve (CUDA events on the solve stream) */
  double relax_kernel_ms;    /* of which: inside the relaxation kernel, summed over its
                                launches (only measured with opts.profile_kernels)         */
  long long relax_launches;  /* launches of the relaxation kernel                          */
  double h2d_ms, d2h_ms;     /* host<->device copies performed by the call                 */
  long long h2d_bytes, d2h_bytes;
  long long units_run;       /* (warp, tile) work units executed by the tiled kernel          */
  long long units_changed;   /* ... of which lowered at least one travel time                 */
} sweeptt_stats;

/* ---- discovery / errors ------------------------------------------------- */

/* cuda/cudasweep-tt-multistart.cu:187-201 (cudaGetDeviceCount + property print). */
int sweeptt_device_count(void);
/* Writes "name, SMs, clock kHz, smem/block optin" for `device`; returns non-zero on success. */
int sweeptt_device_info(int device, char *name, int name_len, int *sm_count, int *clock_khz,
                        size_t *smem_optin);
const char *sweeptt_last_error(void);
const char *sweeptt_version(void);

/* ---- forward star helpers ----------------------------------------------- */

/* serial_new/sweep-tt-multistart.c:120-128: fills fs[l].d = delta*(float)sqrt(i*i+j*j+k*k). */
void sweeptt_star_fill_distances(struct FS *fs, int starsize, float delta);

/* Host-side edge-set analysis (no GPU needed): turns the reference's two-sided
 * "centre relaxes itself and its neighbour" rule with its two quirks
 * (serial_new/...c:160 last offset unused; :219-221 centre==start skipped) into
 * the equivalent pull star.  Outputs (each may be NULL): offsets as (i,j,k)
 * triples, half distances, and a guard flag (1 = this pull is invalid when the
 * neighbour is the start point).  Returns the number of pull offsets, or -1. */
int sweeptt_build_pull_star(const struct FS *fs, int starsize, int star_used, int32_t *ijk_out,
                            float *half_d_out, int32_t *guard_out, int capacity);

/* Test hook (no device needed): how the tiled kernel shares the star's (i,j) columns out between `nw` warps.
 * Columns are grouped by k pattern; kmasks_out[c] is column c's pattern in group order; cuts holds six tables
 * of cut points, cuts[(t * ngroups + g) * (nw + 1) + p] = first column of part p's contiguous piece of group
 * g (entry nw = end of the group).  Returns the number of columns, or -1 if a capacity is too small. */
int sweeptt_debug_column_split(const struct FS *fs, int starsize, int nw, int *ngroups_out,
                               unsigned short *cuts, int cuts_capacity, unsigned *kmasks_out,
                               int kmasks_capacity);

/* ---- one-shot solve: host buffers in, host buffers out -------------------- */

/* Replaces `void cudaRun(int numstart, int starsize)` (cuda/cudasweep-tt-multistart.cu:80,227)
 * and the CPU loop `while(anychange) for s: sweepXYZ(...)` (serial_new/...c:151-170), with
 * explicit arguments instead of the file-scope globals fs[], start[], vbox, ttboxes[].
 * tt_out[s] (nx*ny*nz floats each) receives the converged field of source s; the library
 * initialises travel times itself (INF, 0 at the start; serial_new/...c:139-144).
 * With opts->num_devices > 1 the sources are sharded over the devices with no
 * inter-device communication (the mpi/backup.c:351-363 scheme).
 * More sources than one single-launch solve holds run as consecutive waves; the fields of a finished
 * wave are copied to tt_out[] while the next wave is relaxed.  tt_out[] may be page-locked
 * (sweeptt_host_alloc) or plain malloc memory like the reference's boxalloc; the latter is served
 * through a page-locked stop-over inside the library (the first box decides which way all boxes of a
 * call go; either way is correct for any mix). */
int sweeptt_solve(const float *slowness, int nx, int ny, int nz, const struct FS *fs, int starsize,
                  const struct START *starts, int numstart, float *const *tt_out,
                  const sweeptt_opts *opts, sweeptt_stats *stats);

/* Page-locked host memory for the boxes handed to sweeptt_solve (the counterpart of boxalloc's malloc,
 * include/floatbox.h:122-123): with such buffers the device->host copies of finished sources run at PCIe speed
 * BEHIND the relaxation of the remaining ones; pageable memory works too, only slower (the driver stages it).
 * Returns NULL on failure.  Release with sweeptt_host_free. */
void *sweeptt_host_alloc(size_t bytes);
void sweeptt_host_free(void *p);

/* sweeptt_solve keeps one cached context (device boxes, star tables) per device between
 * calls -- the device-resident float-box pool; this releases them. */
void sweeptt_release_cache(void);

/* ---- device-resident context (float-box pool) ---------------------------- */

/* A context owns one device's padded slowness box, a pool of padded travel-time
 * boxes, the star tables and the convergence state.  It is the device-resident
 * counterpart of the globals vbox/ttboxes[] plus boxalloc/boxsetall/boxput
 * (include/floatbox.h:114-199; device precedent cuda/floatbox.h:194-244). */
typedef struct sweeptt_ctx sweeptt_ctx;

sweeptt_ctx *sweeptt_create(const sweeptt_opts *opts);
void sweeptt_destroy(sweeptt_ctx *ctx);

/* Optional: run all of the context's work on a caller-provided cudaStream_t
 * (passed as void*), e.g. torch's current stream, so the caller's CUDA events see it. */
int sweeptt_set_stream(sweeptt_ctx *ctx, void *cuda_stream);

/* H2D of the slowness box into the padded device box (cuda/...cu:288-294).  Refuses a model
 * with a negative or NaN value (-0.0 is zero), and a model whose kernel axis order the context's
 * star cannot follow (SWEEPTT_KERNEL_TILED: the star, re-ordered, exceeds the tiled kernel's
 * halo); a refused model leaves the context as it was: model, dimensions, star, sources and
 * travel-time boxes.  An accepted model keeps the start points only when its padded size and
 * kernel axis order are the previous model's and every start point lies inside it; otherwise
 * sweeptt_set_sources must be called again before sweeptt_run. */
int sweeptt_set_model(sweeptt_ctx *ctx, const float *slowness, int nx, int ny, int nz);
/* Star tables into __constant__ memory (cuda/...cu:74,285).  Refuses a star in which a used
 * entry (l < starsize-1, or < star_used; the self offset (0,0,0) excepted) has a negative, NaN
 * or infinite d, a star with no usable offset, and, with SWEEPTT_KERNEL_TILED, a star wider than
 * the tiled kernel's halo; a refused star leaves the context as it was. */
int sweeptt_set_star(sweeptt_ctx *ctx, const struct FS *fs, int starsize);
/* Takes numstart boxes from the pool (grows it if needed) and records the start points
 * (serial_new/...c:135-147). Out-of-range starts are an error (the reference would write
 * out of bounds). */
int sweeptt_set_sources(sweeptt_ctx *ctx, const struct START *starts, int numstart);

/* (Re)initialise the travel times on the device and relax to convergence.  Entirely
 * device-resident: no host buffer is touched.  Asynchronous errors surface here.
 *
 * Domain: the kernels' delay fl(0.5f*d * fl(v_n+v_m)) equals the reference's d*(v_n+v_m)/2.0
 * bit for bit only while (dmax, dpos: largest / smallest positive d of the star's used entries;
 * vmax, vpos: largest finite / smallest positive slowness of the model)
 *   fl(dmax * fl(vmax + vmax)) is finite,  every positive d >= 2^-125,  fl(dpos * vpos) >= 2^-125.
 * Outside it this call refuses, with a message naming the bound, and so do sweeptt_step,
 * sweeptt_reset, sweeptt_put_tt, sweeptt_count_violations, the ray and tomography calls,
 * sweeptt_rayset_freeze, the event-location calls, sweeptt_solve and sweeptt_solve_slabs. */
int sweeptt_run(sweeptt_ctx *ctx, sweeptt_stats *stats);

/* Exactly `rounds` relaxation rounds without re-initialising (rounds >= 1); *changed
 * receives 0 when the last round changed nothing.  Used by tests and by profiling. */
int sweeptt_step(sweeptt_ctx *ctx, int rounds, int *changed, sweeptt_stats *stats);
int sweeptt_reset(sweeptt_ctx *ctx); /* INF / 0-at-start re-initialisation only */

/* D2H of one converged box, un-padded into FLOATBOX order (cuda/...cu:393-397). */
int sweeptt_get_tt(sweeptt_ctx *ctx, int source, float *tt_out);
/* H2D of a caller-provided state for source `source` (tests: arbitrary valid upper bounds).  Every value must be
 * +0, positive or +INF: a box holding a NaN, a negative value, -INF or -0.0 is refused with a message naming the
 * first such FLOATBOX index, and the context is left as it was (the scheduling orders times by their bits as
 * unsigned integers, where a set sign bit ranks after +INF; a NaN time would make a location misfit NaN).  A field
 * read back with sweeptt_get_tt never holds -0.0, so it can always be put back. */
int sweeptt_put_tt(sweeptt_ctx *ctx, int source, const float *tt_in);

/* Device-side fixed-point verifier: counts (node, pull offset) pairs that would still
 * lower a travel time (the `testconvergence` invariant,
 * old/wavefront-openmp/wave-multistart.c:300-347, for this edge set). 0 <=> converged. */
int sweeptt_count_violations(sweeptt_ctx *ctx, int source, long long *violations);

/* ---- rays: shortest paths read off a converged field ------------------------ */

/* Status of one traced ray (data, never an error return). */
enum {
  SWEEPTT_RAY_OK = 0,              /* the ray reached the start point                                     */
  SWEEPTT_RAY_UNREACHED = 1,       /* tt[receiver] = +INF                                                  */
  SWEEPTT_RAY_NOT_FIXED_POINT = 2, /* a candidate on the path is below tt[n]: the field is not converged  */
  SWEEPTT_RAY_NO_PREDECESSOR = 3,  /* no candidate equals tt[n]: the field is not of this model/star/start */
  SWEEPTT_RAY_STALLED = 4,         /* the chosen predecessor is not below tt[n] (a zero-delay edge)        */
  SWEEPTT_RAY_TRUNCATED = 5        /* the ray has more than max_nodes nodes; the first max_nodes are kept  */
};

/* Traces, for every source s in [source_begin, source_begin+source_count) and every receiver r, the
 * shortest-path ray from r back to the start point p of s through the field the context holds for s.
 * Receivers are caller-axis node coordinates like start points.
 *
 * Candidate predecessors of a node n != p are exactly the edges the sweep relaxes (o_l: star entries
 * l < star_used): m = n + o_l, and m = n - o_l unless m == p (the reference skips visits whose centre
 * is the start); in-bounds m only.  cand(n,m) = fl(fl(hd*fl(v_n+v_m)) + tt[m]) with hd = 0.5f*d, the
 * sweep's own expression.  At the fixed point every finite tt[n], n != p, equals its smallest candidate.
 * pred(n): among the candidates with cand == tt[n], the one with the smallest tt[m] (-0 before +0),
 * then the one with the smallest FLOATBOX index of m.  The rule depends only on the field and the
 * geometry, never on the relaxation kernel or schedule that produced the field.
 * The ray is r, pred(r), pred(pred(r)), ..., p; a receiver that is the start gives a ray of one node.
 * Its status is SWEEPTT_RAY_UNREACHED when tt[r] = +INF; otherwise the first node n != p of the path at
 * which a candidate is below tt[n] (NOT_FIXED_POINT), no candidate equals tt[n] (NO_PREDECESSOR) or
 * the chosen tt[m] is not below tt[n] (STALLED) ends the ray with that status, n being its last node.
 *
 * Ray (s, r) is stored at q = (s - source_begin)*nrec + r: nodes_out[q*max_nodes + t] (t < length_out[q],
 * caller axes; past the length (-1,-1,-1) up to the call's longest ray, then left as they were), length_out[q], status_out[q] and
 * tt_out[q] = tt[r] (whatever the status: a receiver table without copying whole fields).  Any output
 * may be NULL.  Reads only the model, the field and the start points, so it works after any solve,
 * after sweeptt_step and after sweeptt_put_tt.  Runs on the context's stream and synchronises it.
 * stats (may be NULL): solve_ms = device time of the trace, relaxations = candidate evaluations,
 * kernel_launches, d2h_ms / d2h_bytes. */
int sweeptt_trace_rays(sweeptt_ctx *ctx, int source_begin, int source_count,
                       const struct START *receivers, int nrec, int max_nodes,
                       struct START *nodes_out, /* [source_count*nrec*max_nodes], may be NULL */
                       int32_t *length_out, int32_t *status_out, float *tt_out, /* [source_count*nrec] */
                       sweeptt_stats *stats);

/* ---- tomography: the linear operators of a travel-time inversion over the rays -------- */

/* Both calls trace exactly the rays of sweeptt_trace_rays (same predecessor rule, statuses and max_nodes
 * truncation; ray q = (s - source_begin)*nrec + r) and use only the rays with status SWEEPTT_RAY_OK.  The edges of
 * a ray are its consecutive node pairs (n, m), n nearer the receiver, each with hd = 0.5f*d of its star offset (the
 * sweep's hd).  Nothing but the results leaves the device.  Argument checks, the stream, the synchronisation at the
 * end and stats (solve_ms = device time, relaxations = candidate evaluations, kernel_launches, d2h_ms / d2h_bytes)
 * are those of sweeptt_trace_rays.
 *
 * Projection (G*d): proj_out[q] is the perturbation summed along ray q with the sweep's own expression, from the
 * start point towards the receiver: acc = +0; for each edge from the start end, acc = fl(fl(hd*fl(d_n + d_m)) + acc).
 * A ray of one node gives +0, a ray that is not OK a quiet NaN.  So the projection of the slowness itself equals
 * tt[receiver] bit for bit for every OK ray of a converged field.  Perturbation values are not validated (they
 * propagate per IEEE: -0 sums to +0, d_n + d_m may overflow to INF, INF - INF is NaN).  A NaN result is a quiet NaN
 * with no promised payload or sign.  perturbation: nx*ny*nz floats, FLOATBOX order, caller axes.  Outputs may be NULL. */
int sweeptt_ray_project(sweeptt_ctx *ctx, int source_begin, int source_count,
                        const struct START *receivers, int nrec, int max_nodes,
                        const float *perturbation,          /* nx*ny*nz, FLOATBOX, caller axes */
                        float *proj_out, int32_t *status_out, int32_t *length_out, /* [source_count*nrec], may be NULL */
                        sweeptt_stats *stats);

/* Back-projection (G^T*w): grad[j] = sum over OK rays q, over the edges e of q that touch node j, of w_q*hd_e (an
 * interior node of a ray gets the hd of its two edges, the receiver and the start one each; w = 1 gives the ray
 * coverage).  Exact and deterministic: with hd_max the largest hd of the used star entries, W = max|w_q| and
 * N = source_count*nrec, E is the smallest integer with 2*hd_max*W*N <= 2^(E+62); every contribution
 * c = rint_even(w_q*hd_e*2^-E) (an int64; w*hd is exact in double) is added to both ends of its edge in int64, and
 * grad[j] = S_j*2^E is rounded once to float32 (nearest, ties to even, subnormals included; +-INF from FLT_MAX plus
 * half an ulp on; S_j = 0, contributions that cancel exactly included, gives +0, never -0).  A ray visits a node
 * at most once (travel time strictly decreases along it), so no sum overflows.  *quantum_exp_out = E.  W = 0 (or a
 * star whose hd are all 0) gives all +0 and E = 0.  weights: [source_count*nrec], finite, required; grad_out:
 * nx*ny*nz floats, FLOATBOX order, caller axes, required; quantum_exp_out and status_out may be NULL. */
int sweeptt_ray_backproject(sweeptt_ctx *ctx, int source_begin, int source_count,
                            const struct START *receivers, int nrec, int max_nodes,
                            const float *weights,               /* [source_count*nrec], finite */
                            float *grad_out,                    /* nx*ny*nz, FLOATBOX, caller axes */
                            int *quantum_exp_out, int32_t *status_out, /* may be NULL */
                            sweeptt_stats *stats);

/* ---- ray sets: rays traced once, kept on the device, applied as often as needed -------------- */

/* A linearised inversion step holds the rays fixed and applies G and G^T tens of times; a ray set traces them once.
 *
 * sweeptt_rayset_freeze traces exactly the rays of sweeptt_trace_rays (same predecessor rule, statuses, max_nodes
 * truncation and numbering q = (s - source_begin)*nrec + r; argument checks, stream and synchronisation as there) and
 * keeps, for every OK ray, its steps as pull-table entries (2 bytes each), ray-major in q order.  A ray that is not OK
 * keeps only its status, length and receiver time.  Returns NULL (sweeptt_last_error() set) on any failure, out of
 * device memory included, and then holds nothing.  stats (may be NULL): solve_ms = device time of the trace and the
 * packing, relaxations = candidate evaluations, kernel_launches, d2h_ms / d2h_bytes.
 *
 * Contract: sweeptt_rayset_project and sweeptt_rayset_backproject return bit for bit what sweeptt_ray_project and
 * sweeptt_ray_backproject return for the context state, source range, receivers and max_nodes of the freeze: NaN for
 * a ray that is not OK, +0 for a ray of one node, and the same quantum exponent E (N in its formula is
 * source_count*nrec of the set, rays that are not OK included).
 *
 * The set is a snapshot: it owns copies of the pull table, the geometry and axis permutation, the padded start
 * indices, and its own padded-perturbation, int64-accumulator and staging buffers.  Later set_model, set_star,
 * set_sources, run, step, reset or put_tt calls on the context leave it valid and unchanged.  It borrows only the
 * context's device and stream; its calls run on that stream and synchronise it.  Threading is the context's: use a set
 * from the thread that uses its context, and destroy every set before its context.  The operators read no
 * __constant__ table, so they never wait for another context's star.
 *
 * Device memory (sweeptt_rayset_bytes, not counted in sweeptt_pool_bytes): with N rays, P entries in all, a pull table
 * of npull entries, S = source_count and a padded box of V floats (nx*ny*nz = D nodes),
 *   2*P + 16*N + 8 + 16*npull + 8*S + 12*V + 4*D
 * (entries, offsets int64[N+1], status and one per-ray in/out float, pull table, start indices, perturbation and
 * accumulator boxes, dense staging).  The buffers that freezing needs for a while (the receivers, a chunk of padded
 * records) are the context's grow-only buffers, counted in sweeptt_pool_bytes like those of the other ray calls. */
typedef struct sweeptt_rayset sweeptt_rayset;

sweeptt_rayset *sweeptt_rayset_freeze(sweeptt_ctx *ctx, int source_begin, int source_count,
                                      const struct START *receivers, int nrec, int max_nodes,
                                      sweeptt_stats *stats);
void sweeptt_rayset_destroy(sweeptt_rayset *set);
size_t sweeptt_rayset_bytes(const sweeptt_rayset *set);

/* The per-ray table [source_count*nrec], the values sweeptt_trace_rays returns.  Any output may be NULL. */
int sweeptt_rayset_table(const sweeptt_rayset *set, int32_t *length_out, int32_t *status_out, float *tt_out);

/* Compact node export, decoded on the host from the set's pull table: ray q has the nodes
 * nodes_out[offsets_out[q] .. offsets_out[q+1]) in caller axes, receiver first; only OK rays have nodes (length_q of
 * them), every other ray none.  offsets_out: int64[N+1]; nodes_out: START[offsets_out[N]].  Either may be NULL. */
int sweeptt_rayset_paths(const sweeptt_rayset *set, int64_t *offsets_out, struct START *nodes_out);

/* G*d over every ray of the set (see sweeptt_ray_project).  perturbation: nx*ny*nz floats, FLOATBOX, caller axes of
 * the freeze; proj_out [N] may be NULL.  stats: solve_ms = device time (pad + walk), kernel_launches, d2h. */
int sweeptt_rayset_project(sweeptt_rayset *set, const float *perturbation, float *proj_out, sweeptt_stats *stats);

/* G^T*w over every ray of the set (see sweeptt_ray_backproject).  weights [N] finite, required; grad_out nx*ny*nz
 * floats, required; quantum_exp_out may be NULL.  stats: solve_ms = device time (zeroing, walk, rounding). */
int sweeptt_rayset_backproject(sweeptt_rayset *set, const float *weights, float *grad_out, int *quantum_exp_out,
                               sweeptt_stats *stats);

/* ---- the damped and smoothed least-squares step of a ray set, solved on the device ---------------------------- */

/* sweeptt_rayset_lsqr solves  min ||A x - [b; 0]||^2 + damp^2 ||x||^2,  A = [G_rows; smooth*D],  by LSQR on the device:
 * only b goes to the device (once), only x and a few scalars per iteration come back.
 *
 * G_rows is G over the selected rays (rows[q] != 0; rows NULL = every OK ray; m of them, in q order) with the float32
 * conversions of the set's operators written into it: G_rows x = float64(sweeptt_rayset_project(float32(x)))[rows],
 * G_rows^T y = float64(sweeptt_rayset_backproject(W)), W = float32(y) scattered into [N] with +0 outside rows and the
 * quantum exponent E that sweeptt_rayset_backproject chooses for that W.  Every application is bit for bit what the
 * set's operators return for the same float32 input.
 *
 * D (only when smooth > 0; none at all when smooth = 0) is the first difference: for every caller axis a = 0, 1, 2 in
 * that order and every node n whose neighbour n + e_a is in the box, in FLOATBOX order, one row with the value
 * fl(smooth * fl(x[n+e_a] - x[n])).  Component j of its transpose product is acc = +0; for a = 0, 1, 2: if j - e_a is in
 * the box acc = fl(acc + y_a[j - e_a]), then if j + e_a is in the box acc = fl(acc - y_a[j]); the result is
 * fl(smooth * acc), and A^T y = fl(G part + D part).
 *
 * The algorithm is scipy 1.18's lsqr (scipy/sparse/linalg/_isolve/lsqr.py) statement for statement with x0 = None and
 * calc_var = False, every square a product x*x, in IEEE float64 with no fused multiply-add, except that every
 * np.linalg.norm(v) is sqrt(sumsq(v)) with a fixed order: square every element, pad with +0 to a multiple of 2048,
 * sum every block of 2048 consecutive elements with the halving tree a[i] = fl(a[i] + a[i+h]), h = 1024, 512, .., 1,
 * and apply the same tree to the vector of block sums until one value is left (sumsq of nothing is +0).  The order
 * depends on neither the box, the device nor the grid.  istop, itn and the norms of info mean what scipy's return tuple
 * means.  b = 0 gives x = 0 and istop = 0, as scipy does.  scipy's default iteration limit is 2*nx*ny*nz.
 *
 * Refused with a message before anything runs, the set left as it was: a NULL set; b, opts or x_out NULL; a
 * struct_size of opts (or of info, when given) that is not the sizeof of its struct; rows selecting a ray that is not
 * OK; an element of b that is not finite; damp or smooth negative or not finite; atol, btol or conlim negative or NaN;
 * iter_lim < 0; a star whose edge lengths are not finite; and device memory the workspace cannot get.
 *
 * Device memory: a workspace allocated by the call and freed before it returns, with m selected rows, mD rows of D
 * (smooth > 0: (nx-1)*ny*nz + nx*(ny-1)*nz + nx*ny*(nz-1), else 0) and D = nx*ny*nz nodes,
 *   8*(m + mD) + 24*D + 8*m + 8*(ceil(max(m + mD, D) / 2048) + 1)  bytes
 * (u; x, v and w; the row index int64[m]; the block sums and max|W|), plus 32 bytes of page-locked host memory.
 * The solve uses the set's own perturbation, accumulator, staging and per-ray buffers as scratch, so the set's
 * operators are unchanged afterwards.  It runs on the context's stream and synchronises it; it reads no __constant__
 * table.  stats (may be NULL): solve_ms = elapsed device time of the whole solve (CUDA events; it includes the waits
 * for the host's scalar steps), kernel_launches, h2d_ms / h2d_bytes (b and the row index), d2h_ms / d2h_bytes (the
 * per-iteration scalars and x). */
typedef struct {
  int struct_size;                    /* = sizeof(sweeptt_lsqr_opts)                                         */
  double damp, smooth;                /* finite, >= 0                                                        */
  double atol, btol, conlim;          /* >= 0 (scipy's defaults: 1e-6, 1e-6, 1e8; conlim = 0: no limit)       */
  int iter_lim;                       /* >= 0                                                                */
} sweeptt_lsqr_opts;

typedef struct {
  int struct_size;                    /* = sizeof(sweeptt_lsqr_info)                                         */
  int istop, itn;
  double r1norm, r2norm, anorm, acond, arnorm, xnorm;
} sweeptt_lsqr_info;

int sweeptt_rayset_lsqr(sweeptt_rayset *set, const uint8_t *rows, /* [N] or NULL = the OK rays                  */
                        const double *b,                          /* [number of selected rows], finite           */
                        const sweeptt_lsqr_opts *opts,
                        double *x_out,                            /* nx*ny*nz, FLOATBOX, caller axes of the freeze */
                        sweeptt_lsqr_info *info,                  /* may be NULL                                 */
                        sweeptt_stats *stats);

/* ---- event location: grid search over the stations' travel-time fields ----------------------- */

/* The context's sources [source_begin, source_begin+source_count) are the STATIONS: a field started at a station s
 * gives, by reciprocity, the time from every node n to s.  An event e has source_count picks obs[e][s] (float32, in the
 * units of the fields); NaN means "no pick", every other value must be finite.  P_e = the picked stations in increasing
 * s, k_e = |P_e|.  For every node n (caller axes; j(n) its FLOATBOX index), in IEEE float64, round to nearest, no
 * fused multiply-add, in exactly this order:
 *
 *   if tt_s(n) == +INF for some s in P_e:  misfit = +INF, the node is EXCLUDED
 *   else:
 *     r_s = (double)obs[e][s] - (double)tt_s(n)                 for s in P_e
 *     acc = +0;  for s in P_e ascending: acc = acc + r_s
 *     t0  = acc / (double)k_e
 *     m   = +0;  for s in P_e ascending: u = r_s - t0;  m = m + u*u
 *     misfit = (float)m                                         (one rounding to float32, nearest even)
 *
 * This is least squares with the origin time t0 eliminated.  The two passes keep the misfit >= 0 (the argmin relies
 * on it) and give exactly 0 when all residuals are equal.
 *
 * Best node of e: the node of smallest float32 misfit, ties to the smallest j(n); a node that is not excluded but
 * whose misfit overflows float32 to +INF ranks before every excluded node.  Its origin time is that node's t0.
 * Status (data, never an error return): SWEEPTT_LOC_OK; SWEEPTT_LOC_NO_PICKS when k_e = 0; SWEEPTT_LOC_UNREACHED when
 * every node is excluded.  When the status is not OK: node (-1,-1,-1), misfit +INF, origin NaN; npicks = k_e always.
 *
 * Reciprocity is approximate.  The method uses the station fields as they are.  tt_s(n) can differ slightly from the
 * time of a field started at n: the edge set is not symmetric, because the guarded pull of DESIGN §1 removes the edge
 * {p - o_{L-1}, p} next to each field's own start p.  The contract is the formula above; it claims no exact symmetry.
 *
 * Both calls read only the fields (d_tt) and the geometry, no __constant__ table, so they work after any solve,
 * sweeptt_step or sweeptt_put_tt.  They run on the context's stream and synchronise it.  They refuse, and leave the
 * context as it was, when: the context is not ready (sweeptt_run's checks, the domain guard included); the source
 * range is not within the context's sources; a required output or the picks are NULL; nev < 0; a pick is +INF or
 * -INF; nx*ny*nz > 2^32 (the argmin key holds j(n) in 32 bits); or (sweeptt_locate_events only) source_count exceeds
 * the stations whose times at 32 nodes (8 bytes each) fit the device's opt-in shared memory next to the kernel's
 * static shared memory as cudaFuncGetAttributes reports it: 904 stations on a B200.  The times themselves are not checked here: fields from
 * sweeptt_run / sweeptt_step are +0, positive or +INF, and sweeptt_put_tt refuses anything else.  stats (may be NULL): solve_ms = device time, kernel_launches, h2d_ms / h2d_bytes, d2h_ms / d2h_bytes. */
enum { SWEEPTT_LOC_OK = 0, SWEEPTT_LOC_NO_PICKS = 1, SWEEPTT_LOC_UNREACHED = 2 };

/* picks [nev*source_count], event-major.  best_out (caller-axis node) and status_out are required; misfit_out,
 * origin_out and npicks_out (each [nev]) may be NULL.  The environment variable SWEEPTT_LOCATE_CHUNK (events per
 * launch, default 4096) splits a large nev into several launches; the result does not depend on it. */
int sweeptt_locate_events(sweeptt_ctx *ctx, int source_begin, int source_count, const float *picks, int nev,
                          struct START *best_out, float *misfit_out, double *origin_out,
                          int32_t *npicks_out, int32_t *status_out, sweeptt_stats *stats);

/* The misfit of one event at every node: nx*ny*nz float32 values, FLOATBOX order, caller axes, +INF where excluded
 * (with no pick at all, every node is +0: the formula has no term).  A best node from sweeptt_locate_events is the
 * argmin of this box (ties to the lowest index). */
int sweeptt_misfit_box(sweeptt_ctx *ctx, int source_begin, int source_count, const float *picks /*[source_count]*/,
                       float *misfit_out, sweeptt_stats *stats);

/* The uncertainty of located events: for every event e, the region R_e = { n : misfit_e(n) <= levels[e] } (float32
 * comparison; misfit_e as above), summarised exactly on the device, so that a few dozen numbers per event leave it
 * instead of a misfit box.  Stations, picks [nev*source_count], the per-node formula, the exclusion rule, the
 * refusals, the station limit (the same rule for the call's own kernel: 904 stations on a B200) and the stats are
 * those of sweeptt_locate_events.
 *   - Excluded nodes, and nodes whose misfit overflows float32 to +INF, are never in R_e: for every accepted level R_e
 *     is exactly { n : box[n] <= levels[e] } of the event's sweeptt_misfit_box.  An event with no pick has an empty
 *     region (its misfit box is +0 everywhere: the one exception), and so has a NaN level.
 *   - levels [nev]: NaN, or finite and >= 0.  -0.0 is +0.  +INF, -INF and negative levels are refused, with the
 *     event's index in the message.
 *   - count_out [nev]: |R_e|.  bbox_out [nev*6]: lo0 lo1 lo2 hi0 hi1 hi2, inclusive, caller axes.  moments_out [nev*9]:
 *     S0 S1 S2 S00 S11 S22 S01 S02 S12, the sums over R_e of c_a and c_a*c_b for the caller-axis node coordinates c.
 *     origin_range_out [nev*2]: the smallest and largest origin time t0 over R_e, the formula's t0.  status_out [nev]:
 *     SWEEPTT_LOC_* exactly as sweeptt_locate_events gives it.  An empty region has bbox -1s, moments 0 and origin
 *     range NaN, NaN.  count_out and status_out are required; the others may be NULL.
 *   - Exactness: every output is an integer sum, an integer min / max or a min / max of doubles (compared through the
 *     order-preserving map of their bits to uint64; t0 is never -0, since its sum starts at +0 and a nonzero sum of
 *     float32 differences, at least 2^-149, divided by k <= 2^31 does not underflow).  So every output is bit-identical
 *     for any schedule, chunking (SWEEPTT_LOCATE_CHUNK), kernel that produced the fields or axis permutation.
 *   - A further refusal: a box whose second moments could overflow int64, D * max_a (n_a - 1)^2 > 2^63 - 1 with
 *     D = nx*ny*nz (a line of 2^21 + 1 nodes; 2401 x 2401 x 501 gives 1.7e16), before any allocation. */
int sweeptt_misfit_regions(sweeptt_ctx *ctx, int source_begin, int source_count, const float *picks, int nev,
                           const float *levels, int64_t *count_out, int32_t *bbox_out, int64_t *moments_out,
                           double *origin_range_out, int32_t *status_out, sweeptt_stats *stats);

/* In-bounds pull evaluations of one full round of one source (analytic). */
long long sweeptt_relaxations_per_round(sweeptt_ctx *ctx);
/* Bytes of device memory currently held by the context's pool. */
size_t sweeptt_pool_bytes(sweeptt_ctx *ctx);
/* Tiles (= activation keys) per source of the current model; the single-launch scheduler takes as many
 * sources per launch as fit its shared-memory key snapshot, more sources run as consecutive waves. */
long long sweeptt_tiles_per_source(sweeptt_ctx *ctx);
/* Test hook: what the context keeps of its model's statistics.  vmin = the exact minimum, -0.0 counted as
 * +0.0 (the lower bound of every edge delay that the downwind filter uses; -1 when the model is all +INF and the
 * filter is off); vmax / vpos = the largest finite / smallest positive slowness (the domain of sweeptt_run).
 * Any pointer may be NULL.  Returns 0 without a model. */
int sweeptt_debug_model_stats(sweeptt_ctx *ctx, float *vmin, float *vmax, float *vpos);

/* ---- single huge grid over the devices of one box ----------------------------------------- */

/* Replaces the MPI ghost-cell decomposition (mpi/16partsmpi.c:740-909,
 * mpi/sweep-tt-multistart.c:422-556; ghost width = star radius) for ONE source on ONE grid.
 * opts->num_devices = number of parts (more parts than visible devices share devices round-robin);
 * opts->slab_axis = the caller axis the grid is cut along.  The slowness box and the travel-time box
 * are each one virtual address range whose pages are dealt block-cyclically (blocks of a few tiles
 * along slab_axis) to the devices; every device relaxes the tiles of its own blocks, its TMA loads
 * read halo planes straight from the owner's memory over NVLink and a changed tile wakes its
 * neighbours through the owning device's activation keys.  There are no ghost copies and no exchange
 * step; the host only detects quiescence (opts->rounds_per_poll rounds per look, default 4).
 * The result is bit-identical to the single-device field.  stats->solve_ms is the host wall clock
 * of the relaxation phase, h2d_ms / d2h_ms those of upload (incl. set-up) and gather. */
int sweeptt_solve_slabs(const float *slowness, int nx, int ny, int nz, const struct FS *fs,
                        int starsize, struct START start, float *tt_out, const sweeptt_opts *opts,
                        sweeptt_stats *stats);

/* Same, but every part loads only the planes of its own blocks from the .vbox file with the subset
 * reader (include/velocityboxfiler.h:741) -- what mpi/16partsmpi.c would need for models that do not
 * fit one node's memory.  Model dimensions come from the file header. */
int sweeptt_solve_slabs_vbox(const char *vbox_path, const struct FS *fs, int starsize, struct START start,
                             float *tt_out, const sweeptt_opts *opts, sweeptt_stats *stats);

/* ---- file formats (drop-in surface of the CLI) ---------------------------- */

/* include/velocityboxfiler.h:631 vbfileloadbinary: *slowness is malloc'd (free with
 * sweeptt_free). Fails on bad magic, short file or checksum mismatch (:540-547,:727-732). */
int sweeptt_vbox_load(const char *path, float **slowness, int origin[3], int dims[3]);
/* include/velocityboxfiler.h:511 vbfileopenbinary: header only (dimensions of the stored box). */
int sweeptt_vbox_dims(const char *path, int dims[3]);
/* include/velocityboxfiler.h:310 vbfilestorebinary (byte-identical output). */
int sweeptt_vbox_store(const char *path, const float *slowness, const int origin[3],
                       const int dims[3]);
/* include/velocityboxfiler.h:741 vbfileloadbinarysubset via :511 vbfileopenbinary: reads the
 * sub-box of size sub_dims without reading the rest of the file (checksum not verified, :798-799).
 * sub_origin is FILE-RELATIVE: a 0-based index into the stored box, NOT the absolute coordinates
 * that the reference's bounds check compares with the file's min corner (:761-779, ox >= min);
 * a caller holding absolute coordinates subtracts the origin returned by sweeptt_vbox_load. */
int sweeptt_vbox_load_subset(const char *path, const int sub_origin[3], const int sub_dims[3],
                             float **slowness);
/* Text dialect A "x,y,z,v" per line (include/velocityboxfiler.h:91 vbfileloadtext) and
 * dialect B "nx ny nz" + bare floats (old/wavefront-openmp/wave-multistart.c:151-161);
 * sniffed by the comma on the first line. */
int sweeptt_text_load(const char *path, float **slowness, int origin[3], int dims[3]);
/* serial_new/sweep-tt-multistart.c:111-128: count, then "oi oj ok" rows; d filled with delta. */
int sweeptt_star_load(const char *path, float delta, struct FS **fs, int *starsize);
/* serial_new/sweep-tt-multistart.c:135-147: count, then "si sj sk" rows (0-based). */
int sweeptt_starts_load(const char *path, struct START **starts, int *numstart);
/* serial_new/sweep-tt-multistart.c:176-194: the output.tt text, byte-identical formatting. */
int sweeptt_write_output_tt(const char *path, const float *const *tt, int numstart, int nx, int ny,
                            int nz);
void sweeptt_free(void *p);

#ifdef __cplusplus
}
#endif
#endif /* SWEEPTT_H */
