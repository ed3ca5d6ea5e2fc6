// kernels.h -- host-callable launchers of the sm_100a kernels (kernels.cu).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>

#include "device_types.h"

namespace sweeptt {

struct TiledLaunch {
  int rxy;                   // halo template: 2, 4 or 7
  int stock_id;              // 0 = generic runtime-mask kernel, else a stock-star instantiation
  int nw;                    // compute warps per CTA (the star's columns of a tile are shared out between them)
  int grid;                  // persistent CTAs
  int grid_persistent;       // ... of the single-launch variant
  size_t smem_bytes;
};

// Shared-memory halo variant for a star with max(|i|,|j|) = r (2, 4 or 7), or 0 if none fits.
int tiled_variant_for_radius(int r);
// smem row/plane pitches of a variant (host needs them to precompute column offsets).
void tiled_variant_dims(int rxy, int* sxd, int* syd, int* szd);
// Occupancy-derived persistent grid + opt-in shared memory; returns cudaSuccess or an error.
cudaError_t tiled_prepare(int rxy, int stock_id, int device, TiledLaunch* out);
// Stock-star instantiation whose compile-time pattern list equals `masks` (ascending), or 0.
int tiled_stock_star_for(const uint32_t* masks_ascending, int n, int rxy_needed);

// Upload the column tables into __constant__ memory (stream ordered).
cudaError_t upload_star_constants(const ColumnDev* cols, int ncols, const float* col_hd, int nhd,
                                  const ExtraDev* extra, int nextra, const unsigned* pdesc, int npdesc,
                                  cudaStream_t stream);

struct RelaxArgs {
  BoxGeom g;
  const float* slow;           // padded slowness box
  float* tt;                   // nsrc padded travel-time boxes, contiguous
  int nsrc;
  const int* src_xyz;          // 3 ints per source (logical coords)
  SolveState* st;
  unsigned* worklist;          // 4 * cap entries: one list per generation in flight (round-based scheduling uses two)
  unsigned cap;
  unsigned* key;               // nsrc * ntiles activation keys: float bits of the smallest travel time
                               // that changed next to the tile since it was last relaxed; INF = clean
  unsigned* tmax;              // nsrc * ntiles: float bits of an upper bound of each tile's largest in-grid travel
                               // time (INF until the tile was relaxed with every node reached); nullptr = no filter
  float dmin;                  // lower bound (>= 0) of every edge delay fl(hd*fl(v_n+v_m)) of this model and star
  unsigned* busy;              // nsrc * ntiles: 1 while a tile is on a published list or being relaxed (single-launch
                               // scheduling only: such a tile is never put on a second list)
  unsigned* keysnap;           // nsrc * ntiles scratch words: key snapshot of the generation builder (large problems)
  float bin_scale;             // 32 / bucket (0 when bucket < 0): key -> sort bin of the generation builder
  float bucket;                // only tiles with key <= (smallest key) + bucket run in a round; <0 = all
  const unsigned long long* tile_pulls;  // per tile position: in-bounds pulls of one visit
  int ncols, nextra;
  int max_inner;               // in-tile relaxation passes per visit (>= 1)
  float neg_zero;              // -0.0f passed at run time (see mul2_exact in kernels.cu)
  unsigned lookahead;          // single launch: the list entry this far before the end triggers the next build
  unsigned trig_q8;            // ... but not before this fraction (in 1/256) of the list is handed out
  // ---- one grid spread over several devices (shared_grid.cu): the boxes are ONE virtual address range whose pages
  // live block-cyclically on the devices; every part relaxes the tiles of the x blocks it owns, reads halos from
  // peer memory with the same TMA loads and wakes the owner of a neighbour tile through that part's key array ----
  int nparts;                  // 0 or 1: a single context
  int part;                    // index of this context
  const unsigned char* tx_owner;    // [ntx] owner part of every tile column along x (blocks of a few tiles, dealt round-robin)
  const int* tx_slow0;              // [ntx] owned tiles: first plane of the tile's staged box in this part's local slowness copy
  int slow_pb;                 // != 0: `slow` / the slowness tensor map hold this part's blocks only, each with its halo
                               // planes (slow_pb planes per block, blocks in ascending order)
  unsigned* part_key[MAX_PARTS];    // every part's activation keys (peer memory)
  unsigned* part_tmax[MAX_PARTS];   // every part's per-tile upper bounds (peer memory; nullptr = no filter)
  unsigned* part_kmin[MAX_PARTS];   // every part's published smallest pending key: the activation bucket follows
                                    // the smallest key on ANY device, so no device runs far ahead of the front
  float front_slack;                // ... by more than this (travel-time units; a multiple of the bucket)
  int npat;                    // pattern groups (generic kernel; the stock kernels know theirs at compile time)
  int pat_begin[MAX_PATTERNS + 1];  // stock-star kernels: columns [pat_begin[p], pat_begin[p+1]) share pattern p
};

cudaError_t launch_relax_tiled(const TiledLaunch& tl, const CUtensorMap& tm_slow,
                               const CUtensorMap& tm_tt, const RelaxArgs& a, cudaStream_t stream);
// Single-launch solve: ONE persistent launch relaxes to the fixed point; the CTAs build the next work
// list ("generation") themselves as soon as the current one is handed out, so there is no round barrier,
// no per-round launch and no tail.  Needs launch_reset + launch_persist_begin on the same stream before it.
cudaError_t launch_relax_persistent(const TiledLaunch& tl, const CUtensorMap& tm_slow, const CUtensorMap& tm_tt,
                                    const RelaxArgs& a, cudaStream_t stream);
cudaError_t launch_persist_begin(const RelaxArgs& a, cudaStream_t stream);
cudaError_t launch_persist_check(const RelaxArgs& a, cudaStream_t stream);
size_t tiled_persistent_max_keys(int rxy);
// Two launches: (1) min-reduce the activation keys, (2) move every tile whose key is within the
// bucket of that minimum to the next work list (clearing its key), flip parity, advance the
// round and (when cond != 0) set the CUDA-graph WHILE condition to "work list not empty".
cudaError_t launch_compact(const RelaxArgs& a, unsigned long long cond, cudaStream_t stream);

// Simple (verification / fallback) path: one thread per node and source, global memory.
cudaError_t launch_relax_simple(const RelaxArgs& a, const StarDev* star, int nstar,
                                unsigned long long pulls_per_round, cudaStream_t stream);
cudaError_t launch_advance_simple(SolveState* st, unsigned long long cond, cudaStream_t stream);

// One grid over several devices: the tiles of this part around the start point go on its first work list (reset of
// the shared box itself is done per owned block by the host: launch_fill on plane ranges).
cudaError_t launch_reset_part(const RelaxArgs& a, int max_rounds, cudaStream_t stream);
cudaError_t launch_init_sources(const RelaxArgs& a, cudaStream_t stream);

// Fixed-point verifier.
cudaError_t launch_count_violations(const RelaxArgs& a, int source, const StarDev* star, int nstar,
                                    unsigned long long* out, cudaStream_t stream);

// Ray tracer (include/sweeptt.h, sweeptt_trace_rays): one warp per (source, receiver) pair, source-major.
struct TraceArgs {
  BoxGeom g;
  const float* slow;           // padded slowness box
  const float* tt;             // padded travel-time boxes of the context
  const int* src_xyz;          // 3 ints per source (kernel axes)
  const int* rec_xyz;          // 3 ints per receiver (kernel axes)
  const RayPull* pull;         // npull entries, sorted by kernel-axis (i,j,k)
  int npull;
  int source_begin, nrec;
  long long nrays;             // source_count * nrec
  int max_nodes;
  int* nodes;                  // [nrays * max_nodes * 3] caller-axis node coordinates, or nullptr
  int* length;                 // [nrays]
  int* status;                 // [nrays]
  float* tt_rec;               // [nrays]
  unsigned long long* evals;   // candidate evaluations executed (one counter)
};
size_t trace_rays_smem_bytes(int npull);
cudaError_t launch_trace_rays(const TraceArgs& t, int device, cudaStream_t stream);

// Tomography operators over the same rays (include/sweeptt.h, sweeptt_ray_project / sweeptt_ray_backproject).
// t.nodes and t.tt_rec are unused.
struct TomoArgs {
  TraceArgs t;
  const float* pert;           // projection: padded perturbation box
  float* proj;                 // projection: [nrays] results
  const float* weights;        // back-projection: [nrays] weights
  long long* acc;              // back-projection: padded int64 accumulator box (zeroed by the caller)
  double scale;                // back-projection: 2^-E
  unsigned short* path_global; // per-warp path records in global memory (path_entries entries), or nullptr: in smem
                               // (ray-set record mode: one staging slot of max_nodes entries per ray of the launch)
  long long path_entries;
  long long q_begin;           // ray-set record mode: number of the launch's first ray in the call (t.nrays rays)
};
// Launch shape of a projection or back-projection: persistent grid, dynamic shared memory and where the path
// records live (shared memory when that costs no occupancy; else path_global needs grid * warps * max_nodes entries).
struct RayWalkLaunch {
  int grid;
  size_t smem;
  bool path_in_smem;
  long long path_entries;      // global path entries needed (0 when in smem)
};
cudaError_t ray_walk_prepare(bool backproject, int npull, int max_nodes, long long nrays, int device, RayWalkLaunch* out);
cudaError_t launch_ray_walk(bool backproject, const RayWalkLaunch& l, const TomoArgs& a, cudaStream_t stream);
// Ray sets (include/sweeptt.h, sweeptt_rayset_*).  Record: rays q_begin .. q_begin + t.nrays - 1 traced as by
// the operators, each ray's pull-table entries left in its staging slot a.path_global + q * max_nodes, its length,
// status and receiver time in t.length / t.status / t.tt_rec at q.  Compact: the off[q+1] - off[q] leading entries
// of slot q to dst + off[q].
cudaError_t launch_rayset_record(const TomoArgs& a, int device, cudaStream_t stream);
cudaError_t launch_rayset_compact(const unsigned short* staging, int max_nodes, const long long* off, long long nrays,
                                  unsigned short* dst, cudaStream_t stream);
// G*d or G^T*w over the stored records: a.t supplies g, pull, npull, nrec, nrays and status (the set's); a.pert /
// a.proj or a.weights / a.acc / a.scale as for the operators.
struct RaySetArgs {
  TomoArgs a;
  const long long* offsets;       // [nrays + 1] ray q's entries are entries[offsets[q] .. offsets[q+1])
  const unsigned short* entries;  // pull-table entries of the OK rays, receiver end first (entries_n of them)
  long long entries_n;
  const long long* start_idx;     // [source_count] padded index of every source's start point
};
cudaError_t launch_rayset_walk(bool backproject, const RaySetArgs& s, int device, cudaStream_t stream);
// grad (dense, caller axes) := acc * 2^E rounded once to float32.
cudaError_t launch_grad_finish(const long long* acc, float* dense, BoxGeom g, int E, cudaStream_t stream);

// LSQR over a ray set (include/sweeptt.h, sweeptt_rayset_lsqr).  float64 vectors: u over the m selected rows of G then
// the mD rows of the smoothing operator D, x / v / w over the dense caller-FLOATBOX box.  A launcher whose pass ends
// in a norm leaves sumsq of the pass's outputs in part[0] (the fixed-order block tree, kernels.cu) and adds its
// launches to *launches; the others are one launch each.
struct LsqrArgs {
  long long m, mD;             // rows of G selected, rows of D (0 without smoothing)
  int nx, ny, nz;              // caller axes
  double smooth;
  const long long* row;        // [m] ray of every selected row
  double* u;                   // [m + mD]
  double* x;                   // [D]
  double* v;                   // [D]
  double* w;                   // [D]
  float* io;                   // the set's per-ray floats (projections in, weights out)
  float* stage;                // the set's dense float32 box
  double* part;                // block sums: ceil(max(m + mD, D) / 2048) doubles
  unsigned* wmax;              // bits of max |W| of pass D (zeroed by the caller)
  int ctas;                    // CTAs that share the blocks of a first-level reduction (the result does not depend on it)
};
cudaError_t launch_lsqr_sumsq(const double* p, long long n, double* part, int ctas, cudaStream_t stream, int* launches);
cudaError_t launch_lsqr_to_f32(const double* v, float* stage, long long n, cudaStream_t stream);
cudaError_t launch_lsqr_u(const LsqrArgs& a, double alpha, cudaStream_t stream, int* launches);
cudaError_t launch_lsqr_scale_u(const LsqrArgs& a, double inv_beta, cudaStream_t stream);
cudaError_t launch_lsqr_v(const LsqrArgs& a, double beta, cudaStream_t stream, int* launches);
cudaError_t launch_lsqr_scale(double* p, long long n, double s, cudaStream_t stream);
cudaError_t launch_lsqr_xw(const LsqrArgs& a, double t1, double t2, double inv_rho, cudaStream_t stream, int* launches);

// Event location (include/sweeptt.h, sweeptt_locate_events / sweeptt_misfit_box / sweeptt_misfit_regions).  Event e's picks are entries
// pick_off[e] .. pick_off[e+1] of pick_sta / pick_obs, in increasing station order (NaN picks left out).
struct LocateArgs {
  BoxGeom g;
  const float* tt;             // padded travel-time box of the call's first station; station s at tt + s * g.vol
  int nsta;                    // stations (source_count)
  const int* pick_off;         // [nev + 1]
  const int* pick_sta;         // station of every pick, relative to the first
  const double* pick_obs;      // the pick as a double (exact)
  const double* pick_rk;       // [nev] RN(1.0 / k_e): first guess of the division t0 = acc / k_e (0 when k_e = 0)
  unsigned long long* key;     // [nev] argmin keys (misfit bits << 32 | caller FLOATBOX index), set to ~0 first
  int e_begin, e_count;        // events of one location launch
  int* node;                   // finisher outputs [nev]: caller-axis node (3 ints), misfit, origin time, k_e, status
  float* misfit;
  double* origin;
  int* npicks;
  int* status;
};
// The region slots of sweeptt_misfit_regions (region_kernel, layout in kernels.cu), per event e at [e] or [e * width]:
struct RegionArgs {
  const unsigned* lim;             // level bits + 1 (0: NaN level, no node)
  unsigned long long* sum;         // [10]: count and the 9 moments, zeroed first
  unsigned* box;                   // [6]: min c, min ~c, filled with ones first
  unsigned long long* t0;          // [2]: min key, min ~key of the ordered t0, filled with ones first
  unsigned* reached;               // some node not excluded, zeroed first
};
// Nodes per thread of the location kernel (4, 2 or 1: a CTA stages the times of nsta stations at 32 * that many
// nodes in shared memory), or 0 when not even 32 nodes fit; the same for the region kernel, by its own attributes.
int locate_nodes_per_thread(int nsta, int device);
int region_nodes_per_thread(int nsta, int device);
cudaError_t launch_locate(const LocateArgs& a, int nodes_per_thread, cudaStream_t stream);
// Events [e_begin, e_begin + e_count): the region summaries of sweeptt_misfit_regions.
cudaError_t launch_regions(const LocateArgs& a, const RegionArgs& r, int nodes_per_thread, cudaStream_t stream);
// Decodes every key: best node, and its misfit and t0 recomputed with the location kernel's formula.
cudaError_t launch_locate_finish(const LocateArgs& a, int nev, cudaStream_t stream);
// Event 0's misfit at every node into the dense caller-axis box.
cudaError_t launch_misfit_box(const LocateArgs& a, float* dense, cudaStream_t stream);

// Box utilities (device float-box pool).
cudaError_t launch_fill(float* p, long long n, float value, cudaStream_t stream);
cudaError_t launch_pad_box(const float* dense, float* padded, BoxGeom g, cudaStream_t stream);
cudaError_t launch_unpad_box(const float* padded, float* dense, BoxGeom g, cudaStream_t stream);
// tt := INF everywhere, 0 at each start; state, flags and the first work list reset.
cudaError_t launch_reset(const RelaxArgs& a, int max_rounds, cudaStream_t stream);
// Model statistics, 32 bytes (8-byte aligned): out8[0] = float bits of the smallest slowness of the dense staged
// model (-0.0 counted as +0.0), out8[1] != 0 if any value is negative/NaN, then sum (double) and count (u64) of the
// finite values, out8[6] = bits of the largest finite slowness (0 if none), out8[7] = bits of the smallest positive
// slowness (+INF if none)
cudaError_t launch_min_slowness(const float* dense, long long n, unsigned* out8, cudaStream_t stream);
// tmax[] := INF (call whenever travel times were overwritten from outside, e.g. sweeptt_put_tt)
cudaError_t launch_fill_tmax(const RelaxArgs& a, cudaStream_t stream);
cudaError_t launch_reset_state_only(SolveState* st, int max_rounds, cudaStream_t stream);

}  // namespace sweeptt
