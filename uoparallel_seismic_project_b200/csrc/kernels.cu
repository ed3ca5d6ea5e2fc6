// kernels.cu -- hand-written sm_100a kernels of the multi-start forward-star sweep.
//
// What is computed (arithmetic contract, SURVEY.md §8a): for every node n != start
//     tt[n] = min(tt[n], min over pull offsets o of  fl(fl(hd_o * fl(v_n + v_{n+o})) + tt[n+o]))
// which is the pull form of the reference's two-sided relaxation
// (serial_new/sweep-tt-multistart.c:216,222-249) with hd_o = d_o/2 (exact inside the domain of DESIGN §1) and NO
// fused multiply-add anywhere (__fmul_rn/__fadd_rn never contract; the file is also built
// with -fmad=false).  Any fair relaxation order reaches the same fixed point bit-for-bit,
// because fl(a+c) is monotone in a and travel times only ever decrease.
//
// Kernels
//   relax_tiled<RXY, STAR, NW, PERSIST>
//                     persistent CTAs take tiles (8x8x8 nodes = two 4x8x8 units) from a device work list;
//                     a 2-stage TMA ring (cp.async.bulk.tensor + mbarriers) streams each tile's slowness and
//                     travel-time boxes plus the star-radius halo through shared memory; the star's (i,j)
//                     columns of a unit are shared out between the CTA's warps, each thread owns KZ=8
//                     consecutive z nodes and pulls a 24-float register window of both arrays per column
//                     (LDS.128), running the column's k offsets out of registers with packed fp32x2 math;
//                     the parts meet in per-node min cells in shared memory; changed tiles wake their
//                     neighbours (activation keys, downwind filter); results leave as 128-bit stores.
//                     PERSIST: the whole solve is ONE launch -- the CTAs build the next work list
//                     (build_generation) themselves, ahead of time, while the others keep relaxing.
//   compact_fused / scan_min_key + select_tiles
//                     round-based scheduling: turn the activation keys into the next round's work list,
//                     advance the device-resident round counter and feed the CUDA-graph WHILE condition.
//   relax_simple      one thread per node, global memory, explicit bounds tests: the
//                     verification path and the fallback for stars wider than the halo.
//   count_violations  the fixed-point invariant (testconvergence,
//                     old/wavefront-openmp/wave-multistart.c:300-347) on the device.
//   trace_rays        shortest-path rays from receivers back to the start, read off a converged field
//                     (one warp per ray, exact-match predecessor with a fixed tie rule).
//   ray_project / ray_backproject  the travel-time tomography operators G*d and G^T*w over those rays (the tracer's
//                     predecessor step, then a walk of the recorded path; exact int64 accumulation for G^T*w).
//   rayset_record / rayset_compact / rayset_project / rayset_backproject  ray sets: the same rays traced once and
//                     kept on the device as pull-table entries, then the same walks of the stored records.
//   lsqr_*            the float64 vector passes of a ray set's LSQR solve (conversions, the smoothing stencil, fused
//                     updates) with fixed-order sums of squares.
//   locate / locate_finish / misfit_box  event location: the float64 origin-free least-squares misfit of every
//                     event at every node from the stations' fields, its argmin and the misfit box of one event.
//   fill/pad/unpad/init_sources/min_slowness  the device float-box pool's utilities
//                     (boxsetall/boxput, include/floatbox.h:176-199).
// One grid over several devices (solver.cu, sweeptt_solve_slabs) runs relax_tiled unchanged on a travel-time box
// whose pages live block-cyclically on the devices: halo planes arrive over NVLink through the same TMA loads,
// neighbours on other devices are woken through their owner's key array (RelaxArgs::part_key, tx_owner).
#include "kernels.h"

#include "../../include/sweeptt.h"

#include <cuda_runtime.h>
#include <math_constants.h>

#include <algorithm>
#include <cstdint>
#include <limits>

// -DSWEEPTT_DEBUG_BOUNDS: every TMA coordinate, shared-memory window index, min-cell index, work-list entry and
// result address of the tiled kernel is checked on the device (printf + trap).  compute-sanitizer is not available
// on the GPU pool, so this build run over the random parity cases (tools/debug_bounds.py) is its stand-in.
#ifdef SWEEPTT_DEBUG_BOUNDS
#include <cstdio>
#define DBG_BOUNDS(cond)                                                                                        \
  do {                                                                                                          \
    if (!(cond)) {                                                                                              \
      printf("sweeptt bounds check failed: %s (kernels.cu:%d, block %d, thread %d)\n", #cond, __LINE__, (int)blockIdx.x, \
             (int)(threadIdx.y * blockDim.x + threadIdx.x));                                                    \
      __trap();                                                                                                 \
    }                                                                                                           \
  } while (0)
#else
#define DBG_BOUNDS(cond) do { } while (0)
#endif

namespace sweeptt {

// ---------------------------------------------------------------------------------------
// constant memory: the forward star, column-grouped (cuda/cudasweep-tt-multistart.cu:74
// keeps struct FS dc_fs[] in __constant__; here offsets are pre-resolved to smem offsets
// and the distances are pre-halved)
// ---------------------------------------------------------------------------------------
__constant__ ColumnDev c_cols[MAX_COLUMNS];
__constant__ float c_col_hd[MAX_COL_HD];
__constant__ ExtraDev c_extra[MAX_EXTRA];
// c_pdesc[((xc * 6 + t) * MAX_PATTERNS + g) * MAX_WARPS + p]: the piece of column group g that part p runs, one
// 32-bit constant load per group: first column | (end column << 9) | (index of the first column's first
// half-distance << 18).  Every part walks ALL groups in the same order (instruction-cache locality) and the host
// balances the parts' total cost.  Table t = 0: one live unit shared by all nw warps; t = 1, 2: units 0 and 1
// of a tile with two live units; t = 3..5: the same for the single-launch kernels (their finisher warp needs a
// longer head start).  xc = the tile's position along x: 0 interior, 1 first tile, 2 last tile -- a unit is only 4
// nodes wide, so at the box's x faces whole columns pull from outside the grid for every lane; those tables leave
// them out (on the 241x241x51 box, whose 51 axis is kernel x, that is 7 % of all column evaluations).
__constant__ unsigned c_pdesc[NXCLASS * 6 * MAX_PATTERNS * MAX_WARPS];

cudaError_t upload_star_constants(const ColumnDev* cols, int ncols, const float* col_hd, int nhd,
                                  const ExtraDev* extra, int nextra, const unsigned* pdesc, int npdesc,
                                  cudaStream_t stream) {
  cudaError_t e = cudaSuccess;
  if (npdesc > 0)
    e = cudaMemcpyToSymbolAsync(c_pdesc, pdesc, sizeof(unsigned) * npdesc, 0, cudaMemcpyHostToDevice, stream);
  if (e != cudaSuccess) return e;
  if (ncols > 0)
    e = cudaMemcpyToSymbolAsync(c_cols, cols, sizeof(ColumnDev) * ncols, 0, cudaMemcpyHostToDevice, stream);
  if (e == cudaSuccess && nhd > 0)
    e = cudaMemcpyToSymbolAsync(c_col_hd, col_hd, sizeof(float) * nhd, 0, cudaMemcpyHostToDevice, stream);
  if (e == cudaSuccess && nextra > 0)
    e = cudaMemcpyToSymbolAsync(c_extra, extra, sizeof(ExtraDev) * nextra, 0, cudaMemcpyHostToDevice, stream);
  return e;
}

// ---------------------------------------------------------------------------------------
// PTX helpers: mbarrier + TMA
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE_%=;\n\t"
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t"
      "}" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* tm, uint64_t* bar, int c0, int c1,
                                            int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::
          "r"(smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(tm)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* dst, const CUtensorMap* tm, uint64_t* bar, int c0, int c1,
                                            int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], "
      "[%2];" ::"r"(smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(tm)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}

// ---------------------------------------------------------------------------------------
// tiled relaxation kernel
// ---------------------------------------------------------------------------------------
template <int RXY>
struct TileDims {
  static constexpr int SXD = TX + 2 * RXY;
  static constexpr int SYD = TY + 2 * RXY;
  static constexpr int BOX_FLOATS = SXD * SYD * SZD;
  // every staged box starts on a 128-byte boundary (TMA destination alignment)
  static constexpr int BOX_STRIDE = (BOX_FLOATS * 4 + 127) / 128 * 128 / 4;
  static constexpr int ACC_WORDS = 2 * UNITS * KZ * 32;  // per-node min cells the star's parts are combined through,
                                                         // one set per ring stage (see relax_tiled)
  // 2 pipeline stages x (slowness box + travel-time box) + combine cells + alignment slack
  static constexpr size_t SMEM = sizeof(float) * (4 * BOX_STRIDE + ACC_WORDS) + 128;
};

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// named barriers over the compute warps only (the TMA producer warp never joins them)
__device__ __forceinline__ void named_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
__device__ __forceinline__ void named_arrive(int id, int nthreads) {
  asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
__device__ __forceinline__ int named_sync_or(int id, int nthreads, int pred) {
  int r;
  asm volatile(
      "{\n\t"
      ".reg .pred p, q;\n\t"
      "setp.ne.s32 q, %3, 0;\n\t"
      "bar.red.or.pred p, %1, %2, q;\n\t"
      "selp.s32 %0, 1, 0, p;\n\t"
      "}"
      : "=r"(r)
      : "r"(id), "r"(nthreads), "r"(pred)
      : "memory");
  return r;
}

// ---- column phase -------------------------------------------------------------------------
// One (i,j) column of the star = one 24-float register window of slowness and of travel time
// (LDS.128 granules) + the column's k offsets run out of registers.
template <uint32_t... M>
struct MaskList {};  // compile-time k-pattern list of a stock star; empty = generic kernel

__host__ __device__ constexpr uint32_t granules_of(uint32_t kmask) {
  uint32_t g = 0;
  for (int b = 0; b <= 2 * ZHALO; ++b)
    if (kmask & (1u << b))
      for (int k = 0; k < KZ; ++k) g |= 1u << ((k + b) / 4);
  return g;
}

template <uint32_t GM>
__device__ __forceinline__ void load_window(const float* __restrict__ pv, const float* __restrict__ pt,
                                            float (&W)[WIN], float (&T)[WIN]) {
#pragma unroll
  for (int g = 0; g < WIN / 4; ++g) {
    if (GM & (1u << g)) {
      const float4 wv = *reinterpret_cast<const float4*>(pv + 4 * g);
      const float4 wt = *reinterpret_cast<const float4*>(pt + 4 * g);
      W[4 * g] = wv.x; W[4 * g + 1] = wv.y; W[4 * g + 2] = wv.z; W[4 * g + 3] = wv.w;
      T[4 * g] = wt.x; T[4 * g + 1] = wt.y; T[4 * g + 2] = wt.z; T[4 * g + 3] = wt.w;
    }
  }
}

// ---- packed fp32x2 arithmetic (sm_100: FADD2 / FMUL2) ---------------------------------------
// Two IEEE-754 round-to-nearest fp32 operations per instruction: same bits as the scalar ops,
// half the issue slots.  NEVER an fma: ptxas has been seen to contract mul.rn.f32x2 +
// add.rn.f32x2 into FFMA2 (even with --fmad=false), which would break the bit-exactness
// contract, so the product is produced by fma.rn.f32x2(a, b, -0.0) with a RUNTIME -0.0 operand:
// a*b + (-0) rounds exactly like a*b (signed zeros included) and an FFMA2 cannot be fused into
// the following add.  tests/test_sass.py greps the SASS.
typedef unsigned long long u64;
__device__ __forceinline__ u64 pack2(float lo, float hi) {
  u64 r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
// A pair of consecutive floats read from shared memory at a 4-byte (not 8-byte) aligned address with
// VOLATILE loads: ptxas cannot re-materialise a volatile load, so the pair stays in registers.  Used for
// the odd-aligned slowness pairs (vn[1],vn[2]), ...: built with plain moves, ptxas rebuilds them with two
// MOVs in front of every pattern block's uses (measured: 11 % of all executed instructions).
__device__ __forceinline__ u64 lds_pair_keep(const float* p) {
  float lo, hi;
  const uint32_t addr = smem_u32(p);
  asm volatile("ld.volatile.shared.f32 %0, [%2];\n\tld.volatile.shared.f32 %1, [%2+4];" : "=f"(lo), "=f"(hi) : "r"(addr));
  u64 r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void unpack2(u64 r, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(r));
}
__device__ __forceinline__ u64 add2(u64 a, u64 b) {
  u64 d;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
__device__ __forceinline__ u64 mul2_exact(u64 a, u64 b, u64 negzero2) {
  u64 d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(negzero2));
  return d;
}

__host__ __device__ constexpr int popc_below(uint32_t m, int b) {
  int n = 0;
  for (int i = 0; i < b; ++i) n += (m >> i) & 1u;
  return n;
}

// The arithmetic contract, once: cand = fl(fl(hd * fl(v_n + v_m)) + tt_m); acc = min(acc, cand).
// Node pairs (2j,2j+1) for even window shifts, (2j+1,2j+2) + two scalar ends for odd shifts, so
// that the window operands are always naturally aligned register pairs.  Candidates of two
// consecutive offsets are folded with one 3-input min (FMNMX3).
// candidates of ONE k offset (window shift B = k + ZHALO, compile-time) for the thread's KZ nodes
template <int B>
__device__ __forceinline__ void offset_candidates(const float (&W)[WIN], const float (&T)[WIN], float hd,
                                                  const float (&vn)[KZ], const u64 (&vnE)[KZ / 2],
                                                  const u64 (&vnO)[KZ / 2 - 1], u64 nz2, float (&cand)[KZ]) {
  const u64 hd2 = pack2(hd, hd);
  if constexpr ((B & 1) == 0) {
#pragma unroll
    for (int j = 0; j < KZ / 2; ++j) {
      const u64 sum = add2(vnE[j], pack2(W[2 * j + B], W[2 * j + B + 1]));
      const u64 c2 = add2(mul2_exact(hd2, sum, nz2), pack2(T[2 * j + B], T[2 * j + B + 1]));
      unpack2(c2, cand[2 * j], cand[2 * j + 1]);
    }
  } else {
#pragma unroll
    for (int j = 0; j < KZ / 2 - 1; ++j) {
      const int k = 2 * j + 1;
      const u64 sum = add2(vnO[j], pack2(W[k + B], W[k + B + 1]));
      const u64 c2 = add2(mul2_exact(hd2, sum, nz2), pack2(T[k + B], T[k + B + 1]));
      unpack2(c2, cand[k], cand[k + 1]);
    }
    cand[0] = __fadd_rn(__fmul_rn(hd, __fadd_rn(vn[0], W[B])), T[B]);
    cand[KZ - 1] = __fadd_rn(__fmul_rn(hd, __fadd_rn(vn[KZ - 1], W[KZ - 1 + B])), T[KZ - 1 + B]);
  }
}

template <uint32_t KMASK, int B>
__device__ __forceinline__ void relax_offsets_from(const float (&W)[WIN], const float (&T)[WIN], int& hi,
                                                   const float (&vn)[KZ], const u64 (&vnE)[KZ / 2],
                                                   const u64 (&vnO)[KZ / 2 - 1], u64 nz2, float (&acc)[KZ],
                                                   float (&pend)[KZ]) {
  if constexpr (B <= 2 * ZHALO) {
    if constexpr ((KMASK >> B) & 1u) {
      float cand[KZ];
      offset_candidates<B>(W, T, c_col_hd[hi++], vn, vnE, vnO, nz2, cand);
      if constexpr (popc_below(KMASK, B) & 1) {
#pragma unroll
        for (int k = 0; k < KZ; ++k) acc[k] = fminf(fminf(acc[k], pend[k]), cand[k]);
      } else {
#pragma unroll
        for (int k = 0; k < KZ; ++k) pend[k] = cand[k];
      }
    }
    relax_offsets_from<KMASK, B + 1>(W, T, hi, vn, vnE, vnO, nz2, acc, pend);
  }
}

template <uint32_t KMASK>
__device__ __forceinline__ void relax_column(const float (&W)[WIN], const float (&T)[WIN], int hi,
                                             const float (&vn)[KZ], const u64 (&vnE)[KZ / 2],
                                             const u64 (&vnO)[KZ / 2 - 1], u64 nz2, float (&acc)[KZ]) {
  float pend[KZ];
  relax_offsets_from<KMASK, 0>(W, T, hi, vn, vnE, vnO, nz2, acc, pend);
  if constexpr (popc_below(KMASK, 2 * ZHALO + 1) & 1) {
#pragma unroll
    for (int k = 0; k < KZ; ++k) acc[k] = fminf(acc[k], pend[k]);
  }
}

// generic (runtime-mask) counterpart: one uniform branch per possible k offset
template <int B>
__device__ __forceinline__ void relax_offsets_runtime(uint32_t kmask, const float (&W)[WIN], const float (&T)[WIN],
                                                      int& hi, const float (&vn)[KZ], const u64 (&vnE)[KZ / 2],
                                                      const u64 (&vnO)[KZ / 2 - 1], u64 nz2, float (&acc)[KZ]) {
  if constexpr (B <= 2 * ZHALO) {
    if (kmask & (1u << B)) {
      float cand[KZ];
      offset_candidates<B>(W, T, c_col_hd[hi++], vn, vnE, vnO, nz2, cand);
#pragma unroll
      for (int k = 0; k < KZ; ++k) acc[k] = fminf(acc[k], cand[k]);
    }
    relax_offsets_runtime<B + 1>(kmask, W, T, hi, vn, vnE, vnO, nz2, acc);
  }
}

// The columns of a pattern group share the compile-time k-pattern KMASK (branch-free unrolled block);
// this warp runs ITS piece [lo,hi) of them (descriptor `d`, see c_pdesc).  A group's half-distances are
// contiguous in column order, so their addresses are pure arithmetic.  Window loads are single-buffered:
// with 16 warps per SM the other warps hide the shared-memory latency.
template <uint32_t KMASK>
__device__ __forceinline__ void run_pattern_range(const float* __restrict__ sv, const float* __restrict__ st, int b0,
                                                  const unsigned d, const float (&vn)[KZ],
                                                  const u64 (&vnE)[KZ / 2], const u64 (&vnO)[KZ / 2 - 1], u64 nz2,
                                                  float (&acc)[KZ]) {
  constexpr uint32_t GM = granules_of(KMASK);
  constexpr int NK = popc_below(KMASK, 2 * ZHALO + 1);
  const int lo = (int)(d & 511u), hi_ = (int)((d >> 9) & 511u);
  if (lo >= hi_) return;
  int hi = (int)(d >> 18);
  float W[WIN], T[WIN];
  for (int c = lo; c < hi_; ++c, hi += NK) {
    const int soff = c_cols[c].soff;
    load_window<GM>(sv + b0 + soff, st + b0 + soff, W, T);
    relax_column<KMASK>(W, T, hi, vn, vnE, vnO, nz2, acc);
  }
}

// `f0`: index of this warp's descriptor of group 0 in c_pdesc; `after(g)` runs after pattern group g-1 (the ring feeder's hooks)
template <typename HOOK, uint32_t... M>
__device__ __forceinline__ void columns_phase(MaskList<M...>, const float* __restrict__ sv,
                                              const float* __restrict__ st, int b0, const RelaxArgs& a, int f0,
                                              const float (&vn)[KZ], float (&acc)[KZ], HOOK&& after, int dbg_box_floats) {
  (void)dbg_box_floats;
  u64 vnE[KZ / 2], vnO[KZ / 2 - 1];
#pragma unroll
  for (int j = 0; j < KZ / 2; ++j) vnE[j] = pack2(vn[2 * j], vn[2 * j + 1]);
#pragma unroll
  for (int j = 0; j < KZ / 2 - 1; ++j) vnO[j] = lds_pair_keep(sv + b0 + ZHALO + 2 * j + 1);  // = (vn[2j+1], vn[2j+2])
  const u64 nz2 = pack2(a.neg_zero, a.neg_zero);
#ifdef SWEEPTT_DEBUG_BOUNDS
  {  // every window this warp is going to read lies inside the staged box; every half-distance inside its table
    const int ngroups = sizeof...(M) == 0 ? a.npat : (int)sizeof...(M);
    DBG_BOUNDS(ngroups <= MAX_PATTERNS && f0 >= 0 && f0 + (ngroups - 1) * MAX_WARPS < NXCLASS * 6 * MAX_PATTERNS * MAX_WARPS);
    for (int g = 0; g < ngroups; ++g) {
      const unsigned d = c_pdesc[g * MAX_WARPS + f0];
      const int lo = (int)(d & 511u), hi_ = (int)((d >> 9) & 511u);
      DBG_BOUNDS(lo <= hi_ && hi_ <= a.ncols && a.ncols <= MAX_COLUMNS);
      for (int c = lo; c < hi_; ++c) {
        const ColumnDev col = c_cols[c];
        DBG_BOUNDS(b0 + col.soff >= 0 && b0 + col.soff + WIN <= dbg_box_floats);
        DBG_BOUNDS(col.hd_begin >= 0 && col.hd_begin + __popc(col.kmask) <= MAX_COL_HD);
      }
    }
  }
#endif
  if constexpr (sizeof...(M) == 0) {
    // generic: runtime masks (any star that fits the halo)
    float W[WIN], T[WIN];  // granules a column does not touch keep stale, never-read values
#pragma unroll
    for (int m = 0; m < WIN; ++m) { W[m] = 0.f; T[m] = CUDART_INF_F; }
    for (int g = 0; g < a.npat; ++g) {
      const unsigned d = c_pdesc[g * MAX_WARPS + f0];
      const int lo = (int)(d & 511u), hi_ = (int)((d >> 9) & 511u);
      for (int c = lo; c < hi_; ++c) {
        const ColumnDev col = c_cols[c];
        const float* pv = sv + b0 + col.soff;
        const float* pt = st + b0 + col.soff;
#pragma unroll
        for (int q = 0; q < WIN / 4; ++q) {
          if (col.gmask & (1u << q)) {
            const float4 wv = *reinterpret_cast<const float4*>(pv + 4 * q);
            const float4 wt = *reinterpret_cast<const float4*>(pt + 4 * q);
            W[4 * q] = wv.x; W[4 * q + 1] = wv.y; W[4 * q + 2] = wv.z; W[4 * q + 3] = wv.w;
            T[4 * q] = wt.x; T[4 * q + 1] = wt.y; T[4 * q + 2] = wt.z; T[4 * q + 3] = wt.w;
          }
        }
        int hi = col.hd_begin;
        relax_offsets_runtime<0>(col.kmask, W, T, hi, vn, vnE, vnO, nz2, acc);
      }
      after(g + 1, a.npat);
    }
  } else {
    int g = 0;
    ((run_pattern_range<M>(sv, st, b0, c_pdesc[g * MAX_WARPS + f0], vn, vnE, vnO, nz2, acc),
      ++g, after(g, (int)sizeof...(M))),
     ...);
  }
}

// ---- single-launch scheduling helpers -----------------------------------------------------------
__device__ __forceinline__ unsigned ld_volatile_u32(const unsigned* p) { return *reinterpret_cast<const volatile unsigned*>(p); }
__device__ __forceinline__ void st_volatile_u32(unsigned* p, unsigned v) { *reinterpret_cast<volatile unsigned*>(p) = v; }
__device__ __forceinline__ void fence_proxy_async_all() { asm volatile("fence.proxy.async;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async_global() { asm volatile("fence.proxy.async.global;" ::: "memory"); }

constexpr int GEN_BINS = 32;
constexpr int TILE_NONE = -1;     // staged instead of a tile: the solve is finished
constexpr int TILE_NEXT_GEN = -2; // staged instead of a tile: this generation's list is handed out
constexpr int TILE_BUILD = -3;    // staged instead of a tile: this CTA popped the list's trigger entry and builds the
                                  // next generation EARLY, while the other CTAs are still busy with the rest of the list

// Build generation `g_new` from the activation keys (the device-side counterpart of compact_fused, run by
// ONE CTA while the others keep relaxing): smallest pending key -> bucket threshold -> counting sort of the
// selected tiles by key into work list (g_new & 1).  Tiles that are still on a list or being relaxed
// (busy) are left for a later generation, so a tile is never relaxed by two CTAs at once.  `cache` takes a
// snapshot of the keys (other CTAs keep lowering them while the three passes run): the CTA's idle TMA ring,
// or a global scratch array for problems with more keys than that.  Nothing pending and nothing in flight =
// fixed point.
template <int NCT>
__device__ void build_generation(const RelaxArgs& a, unsigned g_new, unsigned* cache, bool early) {
  __shared__ unsigned s_min, s_inflight, s_stop;
  __shared__ unsigned s_bin[GEN_BINS + 1];
  SolveState* S = a.st;
  const int tid = threadIdx.y * 32 + threadIdx.x;  // (32, NW) blocks
  const unsigned total = (unsigned)((size_t)a.nsrc * a.g.ntx * a.g.nty * a.g.ntz);
  unsigned* wl = a.worklist + (size_t)(g_new & 3u) * a.cap;
  for (unsigned spins = 0;; ++spins) {
    if (tid == 0) {
      s_inflight = atomicAdd(&S->inflight, 0u);  // BEFORE the scan: 0 here means nobody can still add a key
      s_min = 0x7f800000u;
      s_stop = 0u;
    }
    if (tid <= GEN_BINS) s_bin[tid] = 0;
    __syncthreads();
    const unsigned inflight_before = s_inflight;
    unsigned m = 0x7f800000u;
#pragma unroll 16
    for (unsigned i = tid; i < total; i += NCT) {
      unsigned k = __ldcg(&a.key[i]);
      // a busy tile stays pending in global memory -- unless nothing is in flight, in which case the flag is
      // only the not-yet-visible tail of a finished tile (the finish path does not fence for it)
      if (k != 0x7f800000u && inflight_before != 0u && __ldcg(&a.busy[i]) != 0u) k = 0x7f800000u;
      cache[i] = k;
      m = min(m, k);
    }
    m = __reduce_min_sync(0xffffffffu, m);
    if ((tid & 31) == 0 && m != 0x7f800000u) atomicMin(&s_min, m);
    __syncthreads();
    const float kmin = __uint_as_float(s_min);
    const bool all = a.bucket < 0.f;
    const unsigned thr = all ? 0x7f7fffffu : __float_as_uint(kmin + a.bucket);
    const float scale = a.bin_scale;  // GEN_BINS / bucket, divided on the host (a division here would put FFMAs into
                                      // this kernel's SASS, which tests/test_sass.py keeps free of them)
#pragma unroll 8  // (the snapshot may live in global memory: keep several loads in flight)
    for (unsigned i = tid; i < total; i += NCT) {
      const unsigned k = cache[i];
      if (k != 0x7f800000u && k <= thr) {
        const int b = min(GEN_BINS - 1, (int)((__uint_as_float(k) - kmin) * scale));
        atomicAdd(&s_bin[b + 1], 1u);
      }
    }
    __syncthreads();
    if (tid == 0)
      for (int b = 0; b < GEN_BINS; ++b) s_bin[b + 1] += s_bin[b];
    __syncthreads();
    const unsigned cnt = s_bin[GEN_BINS];
    __syncthreads();
#pragma unroll 8
    for (unsigned i = tid; i < total; i += NCT) {
      const unsigned k = cache[i];
      if (k != 0x7f800000u && k <= thr) {
        const int b = min(GEN_BINS - 1, (int)((__uint_as_float(k) - kmin) * scale));
        wl[atomicAdd(&s_bin[b], 1u)] = i;
        a.key[i] = 0x7f800000u;
        a.busy[i] = 1u;
      }
    }
    __threadfence();  // list entries, key and busy updates are visible before the generation is
    __syncthreads();
    if (tid == 0) {
      if (cnt != 0) {
        atomicAdd(&S->inflight, cnt);  // (before the slot: a popped tile can never finish before it is counted)
        atomicExch(&S->gslot[g_new & 3u], (unsigned long long)cnt << 32);  // count | cursor 0, one store
        S->round += 1;
        __threadfence();
        st_volatile_u32(&S->gen, g_new);
        s_stop = 1u;
      } else if (early) {
        st_volatile_u32(&S->builder, g_new - 1u);  // nothing to hand out yet: give the claim back
        s_stop = 1u;
      } else if (s_inflight == 0u) {
        st_volatile_u32(&S->done, 1u);  // fixed point
        s_stop = 1u;
      } else if (spins > (1u << 22)) {
        st_volatile_u32(&S->done, 2u);  // watchdog: tiles in flight never finished
        s_stop = 1u;
      } else {
        __nanosleep(200);  // the tiles in flight will either wake something up or finish
      }
    }
    __syncthreads();
    if (s_stop) break;
  }
}

// Persistent CTA of NW warps.
//   staging   tile ids are popped from the round's work list (one atomicAdd each) and the tile's slowness
//             and travel-time boxes (interior + star-radius halo) are streamed into a 2-stage shared-memory
//             ring with TMA (cp.async.bulk.tensor): tile i+1 lands while tile i is being relaxed.  Thread 0
//             drives the ring from three points of its own column phase, so that neither the atomic nor
//             the work-list load nor the copy is ever waited for.
//   relaxing  a tile is UNITS 4x8x8 units; the star's columns of every live unit are shared out between
//             NW / nlive warps ("parts", cost-balanced cut points from the host), each part keeps its
//             KZ accumulators in registers, lowers the unit's per-node min cells in shared memory
//             (atomicMin on the float bits: travel times are >= 0) and part 0 of the unit (the owner)
//             finishes: start-point pin, changed test, 128-bit stores, activation of the neighbours.
template <int RXY, typename STAR, int NW, bool PERSIST>
// exact block shape (32, NW): threadIdx.y IS the warp index, which lets ptxas treat the per-warp column loops as
// warp-uniform control flow (no BSSY/BSYNC around them)
__global__ void __block_size__((32, NW, 1))
relax_tiled(const __grid_constant__ CUtensorMap tm_slow, const __grid_constant__ CUtensorMap tm_tt,
            const __grid_constant__ RelaxArgs a) {
  using D = TileDims<RXY>;
  constexpr int NCT = 32 * NW;
  // warps with a second duty (the host gives them fewer columns, solver.cu): the unit owners (part 0 of a
  // unit) finish the tile's arithmetic; thread FEED_TID drives the TMA ring; warp FIN_WARP wakes the
  // neighbours and keeps the books
  constexpr int FEED_TID = 32 * (NW / 2 - 1), FIN_WARP = NW - 1;
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  float* ring = reinterpret_cast<float*>(smem_raw + ((128u - (smem_u32(smem_raw) & 127u)) & 127u));
  unsigned* s_acc = reinterpret_cast<unsigned*>(ring + 4 * D::BOX_STRIDE);
  __shared__ __align__(8) uint64_t full[2];
  __shared__ int s_tile[2];
  __shared__ unsigned s_gen;   // PERSIST: the generation this CTA is popping from
  __shared__ int s_role;
  __shared__ unsigned s_tmin;  // float bits of the smallest travel time the tile lowered
  __shared__ unsigned s_tmax;  // float bits of the largest travel time of the tile's in-grid nodes

  const int lane = threadIdx.x;
  const int wq = threadIdx.y;  // warp index
  const int tid = wq * 32 + lane;
  if (tid == 0) {
    mbar_init(&full[0], 1); mbar_init(&full[1], 1);
    fence_mbar_init();
    s_tmin = 0x7f800000u;
    s_tmax = 0u;
    s_gen = 0u;
  }
  for (int i = tid; i < D::ACC_WORDS; i += NCT) s_acc[i] = 0x7f800000u;
  __syncthreads();

  SolveState* S = a.st;
  const int par = S->parity;
  const unsigned cnt = S->count[par];
  const unsigned* wl = a.worklist + (size_t)par * a.cap;
  const int round = S->round;
  const int ntiles = a.g.ntx * a.g.nty * a.g.ntz;

  // stage `q` of the ring <- the boxes of `tile` (or the end marker); thread 0 only
  auto stage_tile = [&](int q, int tile) {
    s_tile[q] = tile;
    if (tile < 0) {
      mbar_arrive(&full[q]);
      return;
    }
    if constexpr (PERSIST) fence_proxy_async_global();  // other CTAs' stores of THIS launch (generic proxy) -> our TMA reads
    const int s = tile / ntiles;
    int tp = tile - s * ntiles;
    const int tz = tp % a.g.ntz; tp /= a.g.ntz;
    const int ty = tp % a.g.nty;
    const int tx = tp / a.g.nty;
    float* sv = ring + q * 2 * D::BOX_STRIDE;
    DBG_BOUNDS(tile >= 0 && s >= 0 && s < a.nsrc && tx >= 0 && tx < a.g.ntx);
    DBG_BOUNDS(tz * TZ + AZ - ZHALO >= 0 && tz * TZ + AZ - ZHALO + SZD <= a.g.pz);
    DBG_BOUNDS(ty * TY + AY - RXY >= 0 && ty * TY + AY - RXY + D::SYD <= a.g.py);
    DBG_BOUNDS(tx * TX + AX - RXY >= 0 && tx * TX + AX - RXY + D::SXD <= a.g.px);
    DBG_BOUNDS(a.slow_pb == 0 || (a.tx_owner[tx] == a.part && a.tx_slow0[tx] >= 0));
    // padded coords of the staged box origin: logical - (RXY, RXY, ZHALO) + apron
    mbar_expect_tx(&full[q], 2u * sizeof(float) * D::BOX_FLOATS);
    int cx = tx * TX + AX - RXY;
    // one grid over several devices: the (read-only) slowness is kept LOCAL -- every owned x block with its own halo
    // planes, slow_pb planes per block, in the order of the part's blocks -- so only travel times cross NVLink
    if (a.slow_pb) cx = a.tx_slow0[tx] + (AX - RXY);
    tma_load_3d(sv, &tm_slow, &full[q], tz * TZ + AZ - ZHALO, ty * TY + AY - RXY, cx);
    tma_load_4d(sv + D::BOX_STRIDE, &tm_tt, &full[q], tz * TZ + AZ - ZHALO, ty * TY + AY - RXY, tx * TX + AX - RXY, s);
  };
  // synchronous pop (prologue, and after a generation switch): next tile id or a marker; thread 0 only
  auto pop_now = [&]() -> int {
    if constexpr (PERSIST) {
      // generations are consumed IN ORDER: a list that was published early must not make anybody leave
      // the rest of the one before it (its tiles would stay busy for ever)
      for (;;) {
        if (ld_volatile_u32(&S->done)) return TILE_NONE;
        const unsigned g = s_gen;
        const unsigned long long w = atomicAdd(&S->gslot[g & 3u], 1ull);  // cursor and count of ONE generation
        const unsigned i = (unsigned)w;
        if (i < (unsigned)(w >> 32)) return (int)__ldcg(&a.worklist[(size_t)(g & 3u) * a.cap + i]);
        if (ld_volatile_u32(&S->gen) == g) return TILE_NEXT_GEN;
        s_gen = g + 1u;
      }
    } else {
      const unsigned i = atomicAdd(&S->cursor, 1u);
      return (i < cnt) ? (int)wl[i] : TILE_NONE;
    }
  };
  if (tid == 0) stage_tile(0, pop_now());

  // lane -> (x within the 4-wide unit, y): a quarter-warp shares x and spans 8 consecutive y, whose
  // rows are SZD = 28 floats apart -> conflict-free LDS.128.
  // Synchronisation of a tile: every warp meets at ONE hardware barrier after its share of the columns
  // (waiting there costs no issue slots; letting the parts run ahead into the next tile's mbarrier spin
  // was measured slower).  Behind it only the unit owners go on with the tile (min cells -> pin -> stores
  // -> neighbour activation) while the other parts already start the next tile, whose min cells are a
  // second set.  With in-tile passes (small stars) every warp takes part in every step.
  const bool multi = a.max_inner > 1;
  const int y = lane & 7;
  bool build_next = false;
  int pend_tile = -1;        // finisher warp, one grid over several devices: tile whose cross-device wake-ups are still to be sent
  unsigned pend_tmin = 0u;
  // A changed node reaches R <= 7 cells: every neighbour tile within that reach may be affected; the tile itself only
  // needs another visit if its last in-tile pass still changed something.  `which`: 0 = every neighbour, 1 = only
  // those owned by this part, 2 = only those owned by other parts.
  auto wake = [&](int wtile, unsigned wtmin, bool wself, int which) {
    const int ws = wtile / ntiles;
    int wp = wtile - ws * ntiles;
    const int wtz = wp % a.g.ntz; wp /= a.g.ntz;
    const int wty = wp % a.g.nty;
    const int wtx = wp / a.g.nty;
    for (int m = lane; m < NMARK; m += 32) {
      const int dx = m / 9 - XREACH, dy = (m / 3) % 3 - 1, dz = m % 3 - 1;
      const int ux = wtx + dx, uy = wty + dy, uz = wtz + dz;
      const bool self = (dx == 0 && dy == 0 && dz == 0);
      bool reach = (abs(dx) - 1) * TX < RXY;  // x distance between the closest nodes of the two tiles
      if (self && !wself) reach = false;
      if (reach && ux >= 0 && ux < a.g.ntx && uy >= 0 && uy < a.g.nty && uz >= 0 && uz < a.g.ntz) {
        const size_t u = (size_t)ws * ntiles + ((size_t)ux * a.g.nty + uy) * a.g.ntz + uz;
        unsigned* keyp = a.key;
        const unsigned* tmaxp = a.tmax;
        if constexpr (!PERSIST) {
          if (a.nparts > 1) {  // the neighbour's x block may belong to another device: its owner keeps its key
            const int o = a.tx_owner[ux];
            if ((which == 1 && o != a.part) || (which == 2 && o == a.part)) continue;
            keyp = a.part_key[o];
            tmaxp = a.part_tmax[o];  // (peer memory for a neighbour elsewhere; measured: dropping the filter there to save the
                                     //  NVLink round trip wakes 4.6 % more tiles and gains nothing)
          }
        }
        // Downwind filter: every candidate that one of our lowered nodes can offer is
        // fl(delay + tt) >= fl(dmin + tmin) (rounding is monotone, delays >= dmin >= 0); a neighbour
        // tile whose nodes are ALL already <= that bound cannot be improved by this change, so it is
        // not woken up.  tmax[] is an upper bound of the tile's current maximum (values only fall).
        bool useful = true;
        if (tmaxp != nullptr && !self)
          useful = __float_as_uint(__fadd_rn(__uint_as_float(wtmin), a.dmin)) < __ldcg(&tmaxp[u]);
        if (useful) atomicMin(&keyp[u], wtmin);
      }
    }
  };
  for (uint32_t it = 0;; ++it) {
    const int q = it & 1;
    mbar_wait(&full[q], (it >> 1) & 1);
    const int tile = s_tile[q];
    if (tile == TILE_NONE) break;
    if constexpr (PERSIST) {
      if (tile == TILE_NEXT_GEN || tile == TILE_BUILD) {
        // TILE_NEXT_GEN: the list of generation s_gen is handed out.  The first CTA to get here builds the
        // next one from the activation keys; CTAs arriving during the build wait for it; later ones find it
        // published.  TILE_BUILD: this CTA builds the next generation ahead of time (nobody waits for it).
        const bool early = tile == TILE_BUILD;
        __syncthreads();  // every warp is done with the previous tile (the ring is idle: it is the build's cache)
        for (;;) {
          if (tid == 0) {
            const unsigned g = s_gen;  // the generation this CTA is in: only its successor is ours to build
            int role = 0;                                                      // 0: nothing to do here
            if (ld_volatile_u32(&S->done)) role = 0;
            else if (ld_volatile_u32(&S->gen) != g) role = 0;                   //    (a newer list is there)
            else if (atomicCAS(&S->builder, g, g + 1u) == g) role = 2;          // 2: build it
            else role = early ? 0 : 1;                                          // 1: wait for the builder
            s_role = role;
          }
          __syncthreads();
          const int role = s_role;
          __syncthreads();
          if (role == 2) {
            // key snapshot: the idle TMA ring when every key fits it, else a global scratch array
          const size_t nkeys = (size_t)a.nsrc * ntiles;
          build_generation<NCT>(a, s_gen + 1u,
                                nkeys <= (size_t)4 * D::BOX_STRIDE ? reinterpret_cast<unsigned*>(ring) : a.keysnap, early);
            fence_proxy_async_all();  // the ring was written through the generic proxy; TMA fills it next
            __syncthreads();
            break;
          }
          if (role == 0) break;
          if (tid == 0) {
            // wait for the builder; an EARLY builder may give its claim back (nothing to hand out yet), then
            // somebody who is out of work -- us -- has to build
            unsigned spins = 0;
            while (ld_volatile_u32(&S->gen) == s_gen && !ld_volatile_u32(&S->done) &&
                   ld_volatile_u32(&S->builder) != s_gen) {
              __nanosleep(100);
              if (++spins > (1u << 24)) { st_volatile_u32(&S->done, 2u); break; }
            }
          }
          __syncthreads();
        }
        if (tid == 0) stage_tile(q ^ 1, pop_now());
        continue;
      }
    }
    // stage q^1 is free (every warp is past the last barrier of the previous tile): claim the next tile.
    // Thread 0 does it in steps spread over its column phase, each consuming what the previous one asked
    // for, so that no atomic, load or copy is ever waited for.
    unsigned pop_i = 0, pop_g = 0, pop_c = 0;
    unsigned long long pop_w = 0;
    int next_tile = TILE_NONE;
    const bool build_now = build_next;  // (feeder thread) the tile staged last time was the list's trigger entry
    build_next = false;
    if (tid == FEED_TID) {
      if constexpr (PERSIST) pop_g = s_gen;
      else pop_i = atomicAdd(&S->cursor, 1u);
    }
    const int s = tile / ntiles;
    int tp = tile - s * ntiles;
    const int tz = tp % a.g.ntz; tp /= a.g.ntz;
    const int ty = tp % a.g.nty;
    const int tx = tp / a.g.nty;
    const int x0 = tx * TX, y0 = ty * TY, z0 = tz * TZ;  // logical coords of the tile interior
    const float* sv = ring + q * 2 * D::BOX_STRIDE;
    float* st = ring + q * 2 * D::BOX_STRIDE + D::BOX_STRIDE;

    // live units (those with nodes inside the grid) and this warp's share of the star
    const int nlive = (UNITS == 2 && x0 + 4 < a.g.nx) ? 2 : 1;
    const int P = NW / nlive;
    const int unit = wq / P, part = wq - unit * P;
    const int xc = tx == 0 ? 1 : (tx == a.g.ntx - 1 ? 2 : 0);  // tile position along x: which columns can reach the grid at all
    // (the finisher of a multi-device part issues system-wide fences like the single-launch kernel's: same head starts)
    int f0 = ((xc * 6 + ((PERSIST || a.nparts > 1) ? 3 : 0) + (nlive == 1 ? 0 : 1 + unit)) * MAX_PATTERNS) * MAX_WARPS + part;  // c_pdesc index, group 0
    // keep the index in ONE register: left alone, ptxas re-derives it (unit / part / table selects, 9 instructions)
    // in front of every one of the 18 pattern blocks of every tile
#ifndef SWEEPTT_NO_PIN
    asm volatile("" : "+r"(f0));
#endif
    const bool owner = part == 0;
    const int x = (unit << 2) | (lane >> 3);
    // smem float index of this thread's window start for the (0,0) column
    const int b0 = ((x + RXY) * D::SYD + (y + RXY)) * SZD;
    const int gx = x0 + x, gy = y0 + y, gz = z0;
    const int px = a.src_xyz[3 * s], py = a.src_xyz[3 * s + 1], pz = a.src_xyz[3 * s + 2];
    unsigned* cell = s_acc + ((q * UNITS + unit) * KZ) * 32 + lane;  // cell[k * 32]
    DBG_BOUNDS(((q * UNITS + unit) * KZ + KZ - 1) * 32 + lane < D::ACC_WORDS && unit < UNITS);
    DBG_BOUNDS(b0 + ZHALO >= 0 && b0 + ZHALO + KZ <= D::BOX_FLOATS);
    float vn[KZ], acc[KZ];
#pragma unroll
    for (int j = 0; j < KZ / 4; ++j) {
      const float4 vv = *reinterpret_cast<const float4*>(sv + b0 + ZHALO + 4 * j);
      const float4 tv = *reinterpret_cast<const float4*>(st + b0 + ZHALO + 4 * j);
      vn[4 * j] = vv.x; vn[4 * j + 1] = vv.y; vn[4 * j + 2] = vv.z; vn[4 * j + 3] = vv.w;
      acc[4 * j] = tv.x; acc[4 * j + 1] = tv.y; acc[4 * j + 2] = tv.z; acc[4 * j + 3] = tv.w;
    }

    // In-tile iterations (block Gauss-Seidel): while the tile's own nodes keep changing, publish the
    // new values to the staged box and relax again against the same halo.  Every pass is a set of
    // valid relaxations, so the fixed point is unchanged.
    // The values a pass started from are NOT kept in registers during the column phase: they are still
    // in the staged box (nobody writes it meanwhile) and are read back for the comparisons.
    int reps = 0;
    int last_pass_changed = 0;
    bool published = false;
    unsigned lowered = 0;  // owner: bit k = node k was lowered by this visit
    for (;;) {
      int pass_changed = 0;
      // Thread 0 feeds the ring from two points of its first pass: the work-list entry is read a few
      // pattern groups after the atomic was issued, the copy starts a few groups later -- neither the
      // atomic nor the load nor the copy is ever waited for.
      const bool feeds = (tid == FEED_TID && reps == 0);
      columns_phase(STAR{}, sv, st, b0, a, f0, vn, acc, [&](int g, int npat) {
        const int h0 = (npat + 5) / 6, h1 = (npat + 2) / 3, h2 = (npat + 1) / 2;
        if (feeds) {
          if constexpr (PERSIST) {
            if (build_now) {
              if (g == h2) stage_tile(q ^ 1, TILE_BUILD);
            } else {
            if (g == h0) pop_w = atomicAdd(&S->gslot[pop_g & 3u], 1ull);
            if (g == h1) {
              pop_i = (unsigned)pop_w; pop_c = (unsigned)(pop_w >> 32);
              // the entry `lookahead` before the list's end is the trigger: whoever pops it builds the next
              // generation right after that tile, so that the new list is out when this one runs dry
              // (short lists: not before the fraction trig_q8/256 of the list is handed out)
              if (a.lookahead != 0u && pop_c >= 64u &&
                  pop_i == max(pop_c > a.lookahead ? pop_c - a.lookahead : 0u, (pop_c * a.trig_q8) >> 8))
                build_next = true;
              if (pop_i >= pop_c && ld_volatile_u32(&S->gen) != pop_g) {
                // this generation is handed out and the next one is already published: take the next tile
                // from it right here (the CTA then never leaves its pipeline); else the CTA goes to the switch
                pop_g += 1u;
                s_gen = pop_g;
                pop_w = atomicAdd(&S->gslot[pop_g & 3u], 1ull);
                pop_i = (unsigned)pop_w; pop_c = (unsigned)(pop_w >> 32);
              }
              next_tile = (pop_i < pop_c) ? (int)__ldcg(&a.worklist[(size_t)(pop_g & 3u) * a.cap + pop_i]) : TILE_NEXT_GEN;
            }
            if (g == h2) stage_tile(q ^ 1, next_tile);
            }
          } else {
            if (g == h0) next_tile = (pop_i < cnt) ? (int)wl[pop_i] : TILE_NONE;
            if (g == h1) stage_tile(q ^ 1, next_tile);
          }
        }
      }, D::BOX_FLOATS);
      float bq[KZ];
#pragma unroll
      for (int j = 0; j < KZ / 4; ++j) {
        const float4 tv = *reinterpret_cast<const float4*>(st + b0 + ZHALO + 4 * j);
        bq[4 * j] = tv.x; bq[4 * j + 1] = tv.y; bq[4 * j + 2] = tv.z; bq[4 * j + 3] = tv.w;
      }
      if (owner) {
        // ---- pulls handled one at a time: guarded (invalid when the neighbour is the start,
        //      serial_new/...c:219-221 with :160) and duplicates ----
        for (int e = 0; e < a.nextra; ++e) {
          const ExtraDev ex = c_extra[e];
          const float* pv = sv + b0 + ZHALO + ex.soff;
          const float* pt = st + b0 + ZHALO + ex.soff;
#pragma unroll
          for (int k = 0; k < KZ; ++k) {
            const bool bad = ex.guarded && (gx + ex.i == px) && (gy + ex.j == py) && (gz + k + ex.k == pz);
            const float delay = __fmul_rn(ex.hd, __fadd_rn(vn[k], pv[k]));
            const float cand = __fadd_rn(delay, pt[k]);
            if (!bad) acc[k] = fminf(acc[k], cand);
          }
        }
      } else {
        // a part that found something lower hands it to the owner through the unit's min cells
#pragma unroll
        for (int k = 0; k < KZ; ++k)
          if (acc[k] < bq[k]) atomicMin(cell + k * 32, __float_as_uint(acc[k]));
      }
      named_sync(1, NCT);
      if (owner) {
#pragma unroll
        for (int k = 0; k < KZ; ++k) {
          const unsigned u = cell[k * 32];
          acc[k] = fminf(acc[k], __uint_as_float(u));
          if (u != 0x7f800000u) cell[k * 32] = 0x7f800000u;
        }
        // the start point itself is never relaxed (serial_new/...c:219-221)
        if (gx == px && gy == py) {
#pragma unroll
          for (int k = 0; k < KZ; ++k)
            if (gz + k == pz) acc[k] = bq[k];
        }
#pragma unroll
        for (int k = 0; k < KZ; ++k)
          if (acc[k] < bq[k]) { pass_changed = 1; lowered |= 1u << k; }
      }
      ++reps;
      if (!multi) break;  // one pass per visit
      last_pass_changed = named_sync_or(3, NCT, pass_changed);  // also: every warp is done reading the staged box
      if (!last_pass_changed || reps >= a.max_inner) break;
      if (owner && pass_changed) {
#pragma unroll
        for (int j = 0; j < KZ / 4; ++j)
          *reinterpret_cast<float4*>(st + b0 + ZHALO + 4 * j) = make_float4(acc[4 * j], acc[4 * j + 1], acc[4 * j + 2], acc[4 * j + 3]);
      }
      published = true;
      named_sync(4, NCT);
      if (!owner) {  // the other parts restart from the published values
#pragma unroll
        for (int j = 0; j < KZ / 4; ++j) {
          const float4 tv = *reinterpret_cast<const float4*>(st + b0 + ZHALO + 4 * j);
          acc[4 * j] = tv.x; acc[4 * j + 1] = tv.y; acc[4 * j + 2] = tv.z; acc[4 * j + 3] = tv.w;
        }
      }
    }

    const bool finisher = wq == FIN_WARP;
    if (!multi && !owner && !finisher) continue;  // this part's work on the tile is done

    const int changed = owner && lowered != 0;
    if (owner) {
      float tmin = CUDART_INF_F;
#pragma unroll
      for (int k = 0; k < KZ; ++k)
        if (lowered & (1u << k)) tmin = fminf(tmin, acc[k]);
      if (changed) {
        float* out = a.tt + (size_t)s * a.g.vol + ((size_t)(gx + AX) * a.g.py + (gy + AY)) * a.g.pz + (gz + AZ);
        DBG_BOUNDS(gx < a.g.nx && gy < a.g.ny && gz < a.g.nz);  // only nodes inside the grid are ever lowered
        DBG_BOUNDS(((size_t)(gx + AX) * a.g.py + (gy + AY)) * a.g.pz + (gz + AZ) + KZ <= (size_t)a.g.vol);
#pragma unroll
        for (int j = 0; j < KZ / 4; ++j)
          *reinterpret_cast<float4*>(out + 4 * j) = make_float4(acc[4 * j], acc[4 * j + 1], acc[4 * j + 2], acc[4 * j + 3]);
      }
      // warp-level reduction of "what changed": travel times are >= 0, so float order == uint order
      const unsigned wmin = __reduce_min_sync(0xffffffffu, __float_as_uint(tmin));
      // largest travel time among this unit's in-grid nodes (the downwind filter below)
      float tmx = 0.f;
      if (gx < a.g.nx && gy < a.g.ny) {
#pragma unroll
        for (int k = 0; k < KZ; ++k)
          if (gz + k < a.g.nz) tmx = fmaxf(tmx, acc[k]);
      }
      const unsigned wmax = __reduce_max_sync(0xffffffffu, __float_as_uint(tmx));
      if (lane == 0) {
        atomicMax(&s_tmax, wmax);
        if (wmin != 0x7f800000u) {
          atomicAdd(&S->units_changed, 1ull);
          atomicMin(&s_tmin, wmin);
        }
      }
    }
    // Hand-over to the finisher warp: with in-tile passes every warp meets once more (also the barrier that
    // ends all reads of the staged boxes there); else the owners only ARRIVE at the finisher's barrier and
    // go straight on to the next tile.
    if (multi) {
      if (published) fence_proxy_async();  // generic-proxy writes to the stage precede the next TMA fill
      (void)named_sync_or(3, NCT, changed);
      if (!finisher) continue;
    } else if (owner) {
      named_arrive(5, 32 * (nlive + 1));
      continue;
    } else {
      named_sync(5, 32 * (nlive + 1));
    }
    const unsigned tile_tmin = s_tmin, tile_tmax = s_tmax;
    const int any = tile_tmin != 0x7f800000u;
    if (!multi) last_pass_changed = any;
    __syncwarp();
    if (lane == 0) {  // the next updates come from owners that first meet this warp at the next tile's barrier
      s_tmin = 0x7f800000u;
      s_tmax = 0u;
    }
    if constexpr (!PERSIST) {
      // One grid over several devices: the wake-ups that cross to ANOTHER device need the tile's stores to be visible
      // system-wide first.  They are sent one tile LATE, from here: by now the previous tile's stores have long
      // drained, so the fence does not wait (issued right behind the stores it cost the finisher warp -- and with it
      // the whole tile -- microseconds).  Wake-ups are only consumed after this launch, so the delay costs nothing.
      if (a.nparts > 1 && pend_tile >= 0) {
        __threadfence_system();
        wake(pend_tile, pend_tmin, false, 2);
        pend_tile = -1;
      }
    }
    if (any) {
      // single launch: the owners' stores (ordered before this point by the owners' barrier) must be visible
      // device-wide before any neighbour is woken up
      if constexpr (PERSIST) {
        __threadfence();
        wake(tile, tile_tmin, last_pass_changed != 0, 0);
      } else if (a.nparts > 1) {
        wake(tile, tile_tmin, last_pass_changed != 0, 1);  // neighbours on this device (consumed after the launch)
        // only tiles at the edge of an ownership block have neighbours elsewhere
        if (a.tx_owner[max(tx - XREACH, 0)] != a.part || a.tx_owner[min(tx + XREACH, a.g.ntx - 1)] != a.part) {
          pend_tile = tile;
          pend_tmin = tile_tmin;
        }
      } else {
        wake(tile, tile_tmin, last_pass_changed != 0, 0);
      }
    }
    if (lane == 31) {
      const int tpos = (tx * a.g.nty + ty) * a.g.ntz + tz;
      if (a.tmax != nullptr) a.tmax[(size_t)s * ntiles + tpos] = tile_tmax;
      atomicAdd(&S->tile_visits, 1ull);
      atomicAdd(&S->units_run, (unsigned long long)(reps * nlive));
      atomicAdd(&S->pulls, a.tile_pulls[tpos] * (unsigned long long)reps);
      if (any) atomicMax(&S->last_changed_round, round + 1);
    }
    if constexpr (PERSIST) {
      // the tile is finished: it may go on a list again, and the in-flight count drops (after the
      // neighbour keys were set, so "nothing pending and nothing in flight" is never seen too early)
      __syncwarp();
      if (lane == 0) {
        st_volatile_u32(&a.busy[tile], 0u);
        if (any) __threadfence();  // the neighbours' keys are set before the count can reach zero
        atomicSub(&S->inflight, 1u);
      }
    }
  }
  if constexpr (!PERSIST) {
    if (pend_tile >= 0) {  // (finisher warp) the last tile's cross-device wake-ups
      __threadfence_system();
      wake(pend_tile, pend_tmin, false, 2);
    }
  }
}

// ---------------------------------------------------------------------------------------
// work-list compaction + device-resident round bookkeeping
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) scan_min_key(const RelaxArgs a) {
  const size_t total = (size_t)a.nsrc * a.g.ntx * a.g.nty * a.g.ntz;
  unsigned m = 0x7f800000u;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x)
    m = min(m, a.key[i]);
  m = __reduce_min_sync(0xffffffffu, m);
  if ((threadIdx.x & 31) == 0 && m != 0x7f800000u) atomicMin(&a.st->kmin_bits, m);
  if (a.nparts > 1) {
    // One grid over several devices: the LAST block publishes this part's smallest pending key and resolves the
    // threshold base once (the smallest key on ANY device -- a stale peer value is older, hence lower: only ever too
    // careful -- but at most front_slack behind our own), so that select_tiles reads one local word instead of
    // every block reading every peer over NVLink.
    __shared__ bool last;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) last = (atomicAdd(&a.st->ticket2, 1u) == gridDim.x - 1);
    __syncthreads();
    if (last && threadIdx.x == 0) {
      __threadfence();
      SolveState* S = a.st;
      S->ticket2 = 0;
      const unsigned own = atomicMin(&S->kmin_bits, 0x7f800000u);  // (read through L2)
      unsigned g = own;
      st_volatile_u32(a.part_kmin[a.part], own);
      for (int q = 0; q < a.nparts; ++q)
        if (q != a.part) g = min(g, ld_volatile_u32(a.part_kmin[q]));
      if (own != 0x7f800000u) g = max(g, __float_as_uint(fmaxf(0.f, __uint_as_float(own) - a.front_slack)));
      S->kmin_bits = g;
    }
  }
}

__global__ void __launch_bounds__(256) select_tiles(const RelaxArgs a, unsigned long long cond) {
  SolveState* S = a.st;
  const int nxt = S->parity ^ 1;
  const size_t total = (size_t)a.nsrc * a.g.ntx * a.g.nty * a.g.ntz;
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  // bucket: keys within `bucket` of the smallest pending key (Dijkstra-like ordering at tile
  // granularity; travel times below the bucket are final, so their tiles are not re-relaxed with
  // inputs that are still going to change)
  const unsigned kmin_bits = S->kmin_bits;  // (one grid over several devices: already the global front, see scan_min_key)
  const float kmin = __uint_as_float(kmin_bits);
  const unsigned thr = (a.bucket < 0.f) ? 0x7f7fffffu : __float_as_uint(kmin + a.bucket);
  const unsigned k = (i < total) ? a.key[i] : 0x7f800000u;
  const bool set = (k != 0x7f800000u) && (k <= thr);
  const unsigned ballot = __ballot_sync(0xffffffffu, set);
  if (ballot) {
    const int lane = threadIdx.x & 31;
    const int leader = __ffs(ballot) - 1;
    unsigned base = 0;
    if (lane == leader) base = atomicAdd(&S->count[nxt], (unsigned)__popc(ballot));
    base = __shfl_sync(0xffffffffu, base, leader);
    if (set) {
      a.worklist[(size_t)nxt * a.cap + base + __popc(ballot & ((1u << lane) - 1))] = (unsigned)i;
      a.key[i] = 0x7f800000u;
    }
  }
  // last block done: flip the lists and advance the round
  __shared__ bool last;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) last = (atomicAdd(&S->ticket, 1u) == gridDim.x - 1);
  __syncthreads();
  if (last && threadIdx.x == 0) {
    __threadfence();
    S->ticket = 0;
    S->cursor = 0;
    S->count[nxt ^ 1] = 0;
    S->parity = nxt;
    S->round += 1;
    S->kmin_bits = 0x7f800000u;
#if __CUDA_ARCH__ >= 900
    if (cond) {
      const bool more = (S->count[nxt] != 0) && (S->max_rounds == 0 || S->round < S->max_rounds);
      cudaGraphSetConditional((cudaGraphConditionalHandle)cond, more ? 1u : 0u);
    }
#endif
  }
}

// ---------------------------------------------------------------------------------------
// simple path: one thread per (node, source), global memory, explicit bounds tests
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ float pull_min_global(const RelaxArgs& a, const float* __restrict__ tt, int x, int y,
                                                 int z, const StarDev* __restrict__ star, int nstar, int px, int py,
                                                 int pz, float cur) {
  const size_t n = ((size_t)(x + AX) * a.g.py + (y + AY)) * a.g.pz + (z + AZ);
  const float vn = a.slow[n];
  float best = cur;
  for (int l = 0; l < nstar; ++l) {
    const StarDev o = star[l];
    const int xo = x + o.i, yo = y + o.j, zo = z + o.k;
    if ((unsigned)xo >= (unsigned)a.g.nx || (unsigned)yo >= (unsigned)a.g.ny || (unsigned)zo >= (unsigned)a.g.nz)
      continue;
    if (o.guarded && xo == px && yo == py && zo == pz) continue;
    const size_t m = ((size_t)(xo + AX) * a.g.py + (yo + AY)) * a.g.pz + (zo + AZ);
    const float delay = __fmul_rn(o.hd, __fadd_rn(vn, a.slow[m]));
    best = fminf(best, __fadd_rn(delay, tt[m]));
  }
  return best;
}

__global__ void __launch_bounds__(128) relax_simple(const RelaxArgs a, const StarDev* __restrict__ star, int nstar,
                                                    unsigned long long pulls_per_round) {
  // z fastest across threads -> coalesced
  // grid.x = nx*ny columns (up to 2^31-1), grid.y = z blocks, grid.z = sources
  const int z = blockIdx.y * blockDim.x + threadIdx.x;
  const int y = blockIdx.x % a.g.ny, x = blockIdx.x / a.g.ny;
  const int s = blockIdx.z;
  int changed = 0;
  if (z < a.g.nz) {
    const int px = a.src_xyz[3 * s], py = a.src_xyz[3 * s + 1], pz = a.src_xyz[3 * s + 2];
    float* tt = a.tt + (size_t)s * a.g.vol;
    if (!(x == px && y == py && z == pz)) {
      const size_t n = ((size_t)(x + AX) * a.g.py + (y + AY)) * a.g.pz + (z + AZ);
      const float cur = tt[n];
      const float best = pull_min_global(a, tt, x, y, z, star, nstar, px, py, pz, cur);
      if (best < cur) {
        tt[n] = best;  // chaotic in-place update: any mix of old/new neighbours is a valid relaxation
        changed = 1;
      }
    }
  }
  if (__syncthreads_or(changed) && threadIdx.x == 0) atomicMax(&a.st->last_changed_round, a.st->round + 1);
  if (blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0 && threadIdx.x == 0) atomicAdd(&a.st->pulls, pulls_per_round);
}

__global__ void advance_simple(SolveState* S, unsigned long long cond) {
  S->round += 1;
#if __CUDA_ARCH__ >= 900
  if (cond) {
    const bool more = (S->last_changed_round == S->round) && (S->max_rounds == 0 || S->round < S->max_rounds);
    cudaGraphSetConditional((cudaGraphConditionalHandle)cond, more ? 1u : 0u);
  }
#endif
}

__global__ void __launch_bounds__(128) count_violations_kernel(const RelaxArgs a, int s,
                                                               const StarDev* __restrict__ star, int nstar,
                                                               unsigned long long* out) {
  const int z = blockIdx.y * blockDim.x + threadIdx.x;
  const int y = blockIdx.x % a.g.ny, x = blockIdx.x / a.g.ny;
  unsigned bad = 0;
  if (z < a.g.nz) {
    const int px = a.src_xyz[3 * s], py = a.src_xyz[3 * s + 1], pz = a.src_xyz[3 * s + 2];
    const float* tt = a.tt + (size_t)s * a.g.vol;
    if (!(x == px && y == py && z == pz)) {
      const size_t n = ((size_t)(x + AX) * a.g.py + (y + AY)) * a.g.pz + (z + AZ);
      const float vn = a.slow[n], cur = tt[n];
      for (int l = 0; l < nstar; ++l) {
        const StarDev o = star[l];
        const int xo = x + o.i, yo = y + o.j, zo = z + o.k;
        if ((unsigned)xo >= (unsigned)a.g.nx || (unsigned)yo >= (unsigned)a.g.ny ||
            (unsigned)zo >= (unsigned)a.g.nz)
          continue;
        if (o.guarded && xo == px && yo == py && zo == pz) continue;
        const size_t m = ((size_t)(xo + AX) * a.g.py + (yo + AY)) * a.g.pz + (zo + AZ);
        const float cand = __fadd_rn(__fmul_rn(o.hd, __fadd_rn(vn, a.slow[m])), tt[m]);
        bad += (cand < cur);
      }
    } else if (tt[((size_t)(x + AX) * a.g.py + (y + AY)) * a.g.pz + (z + AZ)] != 0.0f) {
      bad = 1;
    }
  }
  for (int o = 16; o; o >>= 1) bad += __shfl_xor_sync(0xffffffffu, bad, o);
  if ((threadIdx.x & 31) == 0 && bad) atomicAdd(out, (unsigned long long)bad);
}

// ---------------------------------------------------------------------------------------
// ray tracer (include/sweeptt.h, sweeptt_trace_rays)
// ---------------------------------------------------------------------------------------
// One warp per ray, a grid-stride loop over the (source, receiver) pairs in source-major order, so the rays in
// flight read one source's padded box, which stays in L2.  The pull table is staged once per CTA in shared memory
// (not __constant__: the 32 lanes read 32 different entries).  Per step lane q evaluates entries q, q+32, ... with
// the sweep's exact candidate expression; a warp min-reduction over the key (tt[m] in total order, caller-axis rank)
// of the exact matches picks the predecessor.
constexpr int TRACE_THREADS = 256;
constexpr int RAY_BATCH = 4;  // table entries per lane whose gathers are in flight together

// float -> unsigned with the same order (-0 before +0; no NaN ever reaches a key: cand == tt[n] excludes it)
__device__ __forceinline__ unsigned ordered_bits(float f) {
  const unsigned u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

// Stages the pull table in shared memory (once per CTA).
__device__ __forceinline__ const RayPull* stage_ray_pulls(const TraceArgs& t, int4* s_pull_raw) {
  for (int e = threadIdx.x; e < t.npull; e += blockDim.x) s_pull_raw[e] = reinterpret_cast<const int4*>(t.pull)[e];
  __syncthreads();
  return reinterpret_cast<const RayPull*>(s_pull_raw);
}

// One predecessor step of the warp's ray from node n (kernel axes x,y,z; padded index n; tn = tt[n]; n is not the
// start p): every lane evaluates its share of the pull table, the exact-match key reduction picks pred(n).  Returns
// the status that ends the ray (NOT_FIXED_POINT, NO_PREDECESSOR, STALLED), or -1 after moving (x,y,z,n,tn) to pred(n);
// *eb_out is the table entry of the step, the same on every lane.
__device__ __forceinline__ int ray_pred_step(const TraceArgs& t, const RayPull* s_pull, const float* tt, int px,
                                             int py, int pz, int& x, int& y, int& z, long long& n, float& tn,
                                             int* eb_out, unsigned long long& evals) {
  const unsigned FULL = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  const float vn = t.slow[n];
  bool below = false;
  unsigned long long best = ~0ull;  // (ordered tt[m] << 32) | rank of the best exact match so far
  int be = 0;                       // ... and its table entry
  // batches of RAY_BATCH entries per lane: the gathers of a batch are issued together (predicated, from n
  // itself for pulls that do not count), then evaluated
  for (int e0 = lane; e0 < t.npull; e0 += 32 * RAY_BATCH) {
    RayPull o[RAY_BATCH];
    bool ok[RAY_BATCH];
    float tm[RAY_BATCH], vm[RAY_BATCH];
#pragma unroll
    for (int u = 0; u < RAY_BATCH; ++u) {
      const int e = e0 + 32 * u;
      o[u] = s_pull[min(e, t.npull - 1)];
      const int xo = x + o[u].i, yo = y + o[u].j, zo = z + o[u].k;
      ok[u] = e < t.npull && (unsigned)xo < (unsigned)t.g.nx && (unsigned)yo < (unsigned)t.g.ny &&
              (unsigned)zo < (unsigned)t.g.nz && !((o[u].rank & RAY_GUARD_BIT) && xo == px && yo == py && zo == pz);
      const long long m = n + (ok[u] ? o[u].off : 0);
      DBG_BOUNDS(m >= 0 && m < t.g.vol);
      tm[u] = tt[m];
      vm[u] = t.slow[m];
    }
#pragma unroll
    for (int u = 0; u < RAY_BATCH; ++u) {
      const float cand = __fadd_rn(__fmul_rn(o[u].hd, __fadd_rn(vn, vm[u])), tm[u]);
      evals += ok[u];
      below |= ok[u] && cand < tn;
      const unsigned long long key = ((unsigned long long)ordered_bits(tm[u]) << 32) | (o[u].rank & (RAY_GUARD_BIT - 1u));
      if (ok[u] && cand == tn && key < best) { best = key; be = e0 + 32 * u; }
    }
  }
  if (__any_sync(FULL, below)) return SWEEPTT_RAY_NOT_FIXED_POINT;
  // keys are below ~0 (ordered +INF is 0xff800000), so ~0 means no exact match
  const unsigned mt = __reduce_min_sync(FULL, (unsigned)(best >> 32));
  if (mt == ~0u) return SWEEPTT_RAY_NO_PREDECESSOR;
  const unsigned mr = __reduce_min_sync(FULL, (unsigned)(best >> 32) == mt ? (unsigned)best : ~0u);
  const int w = __ffs(__ballot_sync(FULL, best == (((unsigned long long)mt << 32) | mr))) - 1;
  DBG_BOUNDS(w >= 0 && w < 32);
  const int eb = __shfl_sync(FULL, be, w);
  DBG_BOUNDS(eb >= 0 && eb < t.npull);
  const RayPull o = s_pull[eb];
  x += o.i; y += o.j; z += o.k;
  n += o.off;
  const float tm = tt[n];
  if (!(tm < tn)) return SWEEPTT_RAY_STALLED;
  tn = tm;
  *eb_out = eb;
  return -1;
}

__global__ void __launch_bounds__(TRACE_THREADS) trace_rays_kernel(const TraceArgs t) {
  extern __shared__ int4 s_pull_raw[];
#ifdef SWEEPTT_DEBUG_BOUNDS
  unsigned dyn_smem;
  asm("mov.u32 %0, %%dynamic_smem_size;" : "=r"(dyn_smem));
  DBG_BOUNDS(t.npull >= 1 && t.npull < RAY_MAX_PULLS && (size_t)t.npull * sizeof(RayPull) <= dyn_smem);
#endif
  const RayPull* s_pull = stage_ray_pulls(t, s_pull_raw);
  const unsigned FULL = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  const long long warps = (long long)gridDim.x * (blockDim.x >> 5);
  unsigned long long evals = 0;
  for (long long q = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); q < t.nrays; q += warps) {
    const int sr = (int)(q / t.nrec), r = (int)(q % t.nrec);
    const int s = t.source_begin + sr;
    const int px = t.src_xyz[3 * s], py = t.src_xyz[3 * s + 1], pz = t.src_xyz[3 * s + 2];
    const float* tt = t.tt + (size_t)s * t.g.vol;
    int x = t.rec_xyz[3 * r], y = t.rec_xyz[3 * r + 1], z = t.rec_xyz[3 * r + 2];
    DBG_BOUNDS((unsigned)x < (unsigned)t.g.nx && (unsigned)y < (unsigned)t.g.ny && (unsigned)z < (unsigned)t.g.nz);
    long long n = ((long long)(x + AX) * t.g.py + (y + AY)) * t.g.pz + (z + AZ);
    int* nodes = t.nodes ? t.nodes + (size_t)q * t.max_nodes * 3 : nullptr;
    auto put = [&](int len, int kx, int ky, int kz) {  // node `len` of the ray, written in caller axes
      if (nodes && lane == 0) {
        DBG_BOUNDS(len >= 0 && len < t.max_nodes);
        for (int a = 0; a < 3; ++a)  // caller axis a is kernel axis q with perm[q] == a
          nodes[3 * len + a] = t.g.perm[0] == a ? kx : t.g.perm[1] == a ? ky : kz;
      }
    };
    const float t_rec = tt[n];
    float tn = t_rec;
    int len = 1, status;
    put(0, x, y, z);
    if (tn == CUDART_INF_F) {
      status = SWEEPTT_RAY_UNREACHED;
    } else {
      for (;;) {
        if (x == px && y == py && z == pz) { status = SWEEPTT_RAY_OK; break; }
        int eb;
        status = ray_pred_step(t, s_pull, tt, px, py, pz, x, y, z, n, tn, &eb, evals);
        if (status >= 0) break;
        if (len == t.max_nodes) { status = SWEEPTT_RAY_TRUNCATED; break; }
        put(len, x, y, z);
        ++len;
      }
    }
    if (lane == 0) {
      DBG_BOUNDS(q >= 0 && q < t.nrays && len >= 1 && len <= t.max_nodes);
      t.length[q] = len;
      t.status[q] = status;
      t.tt_rec[q] = t_rec;
    }
  }
  for (int o = 16; o; o >>= 1) evals += __shfl_xor_sync(FULL, evals, o);
  if (lane == 0 && evals) atomicAdd(t.evals, evals);
}

// ---------------------------------------------------------------------------------------
// tomography operators (include/sweeptt.h, sweeptt_ray_project / sweeptt_ray_backproject)
// ---------------------------------------------------------------------------------------
// The same warp-per-ray traversal and predecessor step as trace_rays_kernel, but instead of writing nodes the warp
// records the ray's steps as pull-table entries (16 bits: RAY_MAX_PULLS = 2^15) in a per-warp scratch of max_nodes
// entries, in shared memory behind the pull table when that costs no occupancy, else in a global slot per resident
// warp.  Only once the ray is known to be OK is the record walked, 32 edges per round with every lane on one edge,
// from the start end:
//   projection       acc = fl(fl(hd*fl(d_n + d_m)) + acc) from acc = +0, the sweep's own sum in the sweep's order
//                    (sequential: one shuffle + add per edge; the gathers of the chunk are lane-parallel);
//   back-projection  every node of the ray gets rint_even(w*hd*2^-E) of each of its (one or two) edges, added as
//                    int64 atomics into a padded accumulator box: integer sums do not depend on the order, so the
//                    result is deterministic.
// Every ray ends at its start node, so the atomics there contend; they are not aggregated per warp or CTA because the
// back-projection measured no slower than the projection (DESIGN §4d).

// Walks the recorded path of the warp's OK ray from the start end.  Round c gives lane j edge k = nedge-1-(32c+j)
// (live when k >= 0): its table entry e, and the padded indices of its ends n_k (nearer the receiver) and n_{k+1}.
template <class F>
__device__ __forceinline__ void walk_ray_path(const unsigned short* path, int nedge, long long n_start,
                                              const RayPull* s_pull, int npull, F&& f) {
  const unsigned FULL = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  long long cur = n_start;  // n_{k+1} of lane 0's edge
  for (int base = 0; base < nedge; base += 32) {
    const int k = nedge - 1 - (base + lane);
    const bool live = k >= 0;
    const int e = live ? path[k] : 0;
    DBG_BOUNDS(e >= 0 && e < npull);
    const long long o = live ? s_pull[e].off : 0;
    long long sum = o;  // inclusive prefix sum of the offsets over the lanes: n_k = cur - sum
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const long long v = __shfl_up_sync(FULL, sum, d);
      if (lane >= d) sum += v;
    }
    f(live, k, e, cur - sum, cur - sum + o);
    cur -= __shfl_sync(FULL, sum, 31);
  }
}

__device__ __forceinline__ float project_ray(const TomoArgs& a, const RayPull* s_pull, const unsigned short* path,
                                             int nedge, long long n_start) {
  const unsigned FULL = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  float acc = 0.f;
  float d_far = a.pert[n_start];  // perturbation at n_{k+1} of lane 0's edge
  walk_ray_path(path, nedge, n_start, s_pull, a.t.npull, [&](bool live, int k, int e, long long n, long long m) {
    DBG_BOUNDS(!live || (n >= 0 && n < a.t.g.vol && m >= 0 && m < a.t.g.vol));
    const float dn = live ? a.pert[n] : 0.f;
    float dm = __shfl_up_sync(FULL, dn, 1);
    if (lane == 0) dm = d_far;
    const float term = live ? __fmul_rn(s_pull[e].hd, __fadd_rn(dn, dm)) : 0.f;
    const int nlive = min(32, k + lane + 1);  // lanes of this round with an edge (k + lane = nedge-1-base)
    for (int j = 0; j < nlive; ++j) acc = __fadd_rn(__shfl_sync(FULL, term, j), acc);
    d_far = __shfl_sync(FULL, dn, 31);
  });
  return acc;
}

__device__ __forceinline__ long long backproject_quantum(float w, float hd, double scale) {
  // w*hd is exact in double (24 x 24 bits), the power-of-two scale is exact unless the product underflows, which
  // happens only far below 1/2 (rounds to 0 either way)
  return __double2ll_rn(__dmul_rn(__dmul_rn((double)w, (double)hd), scale));
}

__device__ __forceinline__ void backproject_ray(const TomoArgs& a, const RayPull* s_pull, const unsigned short* path,
                                                int nedge, long long n_start, float w) {
  const int lane = threadIdx.x & 31;
  if (lane == 0 && nedge > 0) {  // the start node: its one in-edge
    DBG_BOUNDS(path[nedge - 1] < a.t.npull && n_start >= 0 && n_start < a.t.g.vol);
    const long long c = backproject_quantum(w, s_pull[path[nedge - 1]].hd, a.scale);
    if (c) atomicAdd(reinterpret_cast<unsigned long long*>(a.acc + n_start), (unsigned long long)c);
  }
  walk_ray_path(path, nedge, n_start, s_pull, a.t.npull, [&](bool live, int k, int e, long long n, long long) {
    if (!live) return;
    // node n_k gets edge k and, unless it is the receiver, edge k-1
    long long c = backproject_quantum(w, s_pull[e].hd, a.scale);
    if (k > 0) {
      DBG_BOUNDS(path[k - 1] < a.t.npull);
      c += backproject_quantum(w, s_pull[path[k - 1]].hd, a.scale);
    }
    DBG_BOUNDS(n >= 0 && n < a.t.g.vol);
    if (c) atomicAdd(reinterpret_cast<unsigned long long*>(a.acc + n), (unsigned long long)c);
  });
}

// What the walk body does with a traced ray: the two operators, or (ray sets) keep its record.
enum { WALK_PROJECT = 0, WALK_BACKPROJECT = 1, WALK_RECORD = 2 };

// WALK_RECORD (sweeptt_rayset_freeze): the launch covers rays a.q_begin .. a.q_begin + t.nrays - 1 of the call; ray
// q_begin + q leaves its record in staging slot q (a.path_global + q * max_nodes), its length, status and receiver
// time at index q, and nothing is walked.
template <int MODE>
__device__ __forceinline__ void ray_walk_body(const TomoArgs& a, int4* smem) {
  const TraceArgs& t = a.t;
#ifdef SWEEPTT_DEBUG_BOUNDS
  unsigned dyn_smem;
  asm("mov.u32 %0, %%dynamic_smem_size;" : "=r"(dyn_smem));
  DBG_BOUNDS(t.npull >= 1 && t.npull < RAY_MAX_PULLS && t.max_nodes >= 1 &&
             (size_t)t.npull * sizeof(RayPull) + (a.path_global ? 0 : (size_t)(TRACE_THREADS / 32) * t.max_nodes * 2) <= dyn_smem);
#endif
  const RayPull* s_pull = stage_ray_pulls(t, smem);
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const long long slot = (long long)blockIdx.x * (blockDim.x >> 5) + warp;
  DBG_BOUNDS(MODE == WALK_RECORD || !a.path_global || (slot + 1) * t.max_nodes <= a.path_entries);
  unsigned short* path = MODE == WALK_RECORD ? nullptr
                        : a.path_global      ? a.path_global + slot * t.max_nodes
                                             : reinterpret_cast<unsigned short*>(smem + t.npull) + (size_t)warp * t.max_nodes;
  const long long warps = (long long)gridDim.x * (blockDim.x >> 5);
  unsigned long long evals = 0;
  for (long long q = slot; q < t.nrays; q += warps) {
    const long long qr = MODE == WALK_RECORD ? a.q_begin + q : q;  // the ray's number in the call
    const int sr = (int)(qr / t.nrec), r = (int)(qr % t.nrec);
    const int s = t.source_begin + sr;
    const int px = t.src_xyz[3 * s], py = t.src_xyz[3 * s + 1], pz = t.src_xyz[3 * s + 2];
    const float* tt = t.tt + (size_t)s * t.g.vol;
    int x = t.rec_xyz[3 * r], y = t.rec_xyz[3 * r + 1], z = t.rec_xyz[3 * r + 2];
    DBG_BOUNDS((unsigned)x < (unsigned)t.g.nx && (unsigned)y < (unsigned)t.g.ny && (unsigned)z < (unsigned)t.g.nz);
    long long n = ((long long)(x + AX) * t.g.py + (y + AY)) * t.g.pz + (z + AZ);
    if (MODE == WALK_RECORD) {
      DBG_BOUNDS(a.path_global && (q + 1) * t.max_nodes <= a.path_entries);
      path = a.path_global + q * t.max_nodes;
    }
    const float w = MODE == WALK_BACKPROJECT ? a.weights[q] : 0.f;
    const float t_rec = tt[n];
    float tn = t_rec;
    int len = 1, status;
    __syncwarp();  // the previous ray's walk has read its record
    if (tn == CUDART_INF_F) {
      status = SWEEPTT_RAY_UNREACHED;
    } else {
      for (;;) {
        if (x == px && y == py && z == pz) { status = SWEEPTT_RAY_OK; break; }
        int eb;
        status = ray_pred_step(t, s_pull, tt, px, py, pz, x, y, z, n, tn, &eb, evals);
        if (status >= 0) break;
        if (len == t.max_nodes) { status = SWEEPTT_RAY_TRUNCATED; break; }
        if (lane == 0) {
          DBG_BOUNDS(len - 1 >= 0 && len - 1 < t.max_nodes);
          path[len - 1] = (unsigned short)eb;
        }
        ++len;
      }
    }
    __syncwarp();  // the record is visible to every lane
    if (MODE == WALK_BACKPROJECT) {
      if (status == SWEEPTT_RAY_OK && w != 0.f) backproject_ray(a, s_pull, path, len - 1, n, w);
    } else if (MODE == WALK_PROJECT) {
      const float v = status == SWEEPTT_RAY_OK ? project_ray(a, s_pull, path, len - 1, n) : CUDART_NAN_F;
      if (lane == 0) {
        DBG_BOUNDS(q >= 0 && q < t.nrays);
        a.proj[q] = v;
      }
    }
    if (lane == 0) {
      DBG_BOUNDS(q >= 0 && q < t.nrays && len >= 1 && len <= t.max_nodes);
      t.length[q] = len;
      t.status[q] = status;
      if (MODE == WALK_RECORD) t.tt_rec[q] = t_rec;
    }
  }
  for (int o = 16; o; o >>= 1) evals += __shfl_xor_sync(0xffffffffu, evals, o);
  if (lane == 0 && evals) atomicAdd(t.evals, evals);
}

__global__ void __launch_bounds__(TRACE_THREADS) ray_project_kernel(const TomoArgs a) {
  extern __shared__ int4 s_tomo_raw[];
  ray_walk_body<WALK_PROJECT>(a, s_tomo_raw);
}

__global__ void __launch_bounds__(TRACE_THREADS) ray_backproject_kernel(const TomoArgs a) {
  extern __shared__ int4 s_tomo_raw[];
  ray_walk_body<WALK_BACKPROJECT>(a, s_tomo_raw);
}

// ---------------------------------------------------------------------------------------
// ray sets (include/sweeptt.h, sweeptt_rayset_*)
// ---------------------------------------------------------------------------------------
// Freezing traces a bounded chunk of rays at a time with the walk body in record mode (every ray's record in a staging
// slot of max_nodes entries), then rayset_compact_kernel packs the records of the chunk's OK rays ray-major in q order.
// Applying the set walks the stored records with the operators' own project_ray / backproject_ray: no predecessor is
// picked again, and no __constant__ table is read.
// (4 CTAs per SM, as the tracer has: with no minimum ptxas settles on 48 registers and spills 8 bytes)
__global__ void __launch_bounds__(TRACE_THREADS, 4) rayset_record_kernel(const TomoArgs a) {
  extern __shared__ int4 s_tomo_raw[];
  ray_walk_body<WALK_RECORD>(a, s_tomo_raw);
}

// One warp per ray of the chunk: the nedge = off[q+1] - off[q] leading entries of staging slot q go to dst + off[q].
__global__ void __launch_bounds__(TRACE_THREADS) rayset_compact_kernel(const unsigned short* __restrict__ staging,
                                                                      int max_nodes, const long long* __restrict__ off,
                                                                      long long nrays, unsigned short* __restrict__ dst) {
  const int lane = threadIdx.x & 31;
  const long long warps = (long long)gridDim.x * (blockDim.x >> 5);
  for (long long q = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); q < nrays; q += warps) {
    const long long b = off[q], nedge = off[q + 1] - b;
    DBG_BOUNDS(b >= 0 && nedge >= 0 && nedge < max_nodes && b + nedge <= off[nrays]);
    for (long long j = lane; j < nedge; j += 32) dst[b + j] = staging[q * max_nodes + j];
  }
}

template <bool BACK>
__device__ __forceinline__ void rayset_walk_body(const RaySetArgs& s, int4* smem) {
  const TomoArgs& a = s.a;
  const TraceArgs& t = a.t;
#ifdef SWEEPTT_DEBUG_BOUNDS
  unsigned dyn_smem;
  asm("mov.u32 %0, %%dynamic_smem_size;" : "=r"(dyn_smem));
  DBG_BOUNDS(t.npull >= 1 && t.npull < RAY_MAX_PULLS && (size_t)t.npull * sizeof(RayPull) <= dyn_smem);
#endif
  const RayPull* s_pull = stage_ray_pulls(t, smem);
  const int lane = threadIdx.x & 31;
  const long long warps = (long long)gridDim.x * (blockDim.x >> 5);
  for (long long q = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); q < t.nrays; q += warps) {
    const bool ok = t.status[q] == SWEEPTT_RAY_OK;
    const long long b = s.offsets[q];
    const int nedge = (int)(s.offsets[q + 1] - b);
    const int sr = (int)(q / t.nrec);
    const long long n_start = s.start_idx[sr];
    DBG_BOUNDS(b >= 0 && nedge >= 0 && b + nedge <= s.entries_n && (ok || nedge == 0));
    DBG_BOUNDS(sr >= 0 && (long long)sr * t.nrec < t.nrays && n_start >= 0 && n_start < t.g.vol);
    const unsigned short* path = s.entries + b;
    if (BACK) {
      const float w = a.weights[q];
      if (ok && w != 0.f) backproject_ray(a, s_pull, path, nedge, n_start, w);
    } else {
      const float v = ok ? project_ray(a, s_pull, path, nedge, n_start) : CUDART_NAN_F;
      if (lane == 0) a.proj[q] = v;
    }
  }
}

__global__ void __launch_bounds__(TRACE_THREADS) rayset_project_kernel(const RaySetArgs s) {
  extern __shared__ int4 s_tomo_raw[];
  rayset_walk_body<false>(s, s_tomo_raw);
}

__global__ void __launch_bounds__(TRACE_THREADS) rayset_backproject_kernel(const RaySetArgs s) {
  extern __shared__ int4 s_tomo_raw[];
  rayset_walk_body<true>(s, s_tomo_raw);
}

// grad (dense, caller axes) := S * 2^E rounded once to float32 (nearest, ties to even), S the int64 accumulator
// (padded kernel layout).  Normal results: __ll2float_rn is the one rounding (to 24 bits) and the power-of-two
// scaling after it is exact or overflows exactly when the rounded value does.  Results below 2^-126: the quantum
// is 2^-149, so S is shifted to that quantum with one round-half-even on the integer and stored as the subnormal
// (or smallest normal) it encodes.
__device__ __forceinline__ float round_scaled(long long S, int E) {
  if (S == 0) return 0.f;
  const unsigned sign = S < 0 ? 0x80000000u : 0u;
  const unsigned long long u = S < 0 ? 0ull - (unsigned long long)S : (unsigned long long)S;
  const int lim = -126 - E;  // |S| * 2^E < 2^-126  <=>  |S| < 2^lim
  if (lim > 0 && (lim >= 64 || u < (1ull << lim))) {
    const int sh = -(E + 149);  // S * 2^E = S * 2^-sh quanta of 2^-149
    unsigned long long qv;
    if (sh <= 0) {
      qv = u << -sh;  // < 2^23: exact
    } else if (sh >= 64) {
      qv = 0;         // u < 2^63 <= half a quantum
    } else {
      qv = u >> sh;
      const unsigned long long rem = u & ((1ull << sh) - 1), half = 1ull << (sh - 1);
      if (rem > half || (rem == half && (qv & 1))) ++qv;
    }
    return __uint_as_float(sign | (unsigned)qv);  // qv <= 2^23: subnormal, zero or 2^-126
  }
  return scalbnf(__ll2float_rn(S), E);
}

__global__ void grad_finish_kernel(const long long* __restrict__ acc, float* __restrict__ dense, BoxGeom g, int E) {
  const long long vol = (long long)g.nx * g.ny * g.nz;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < vol; i += (long long)gridDim.x * blockDim.x) {
    const int z = (int)(i % g.nz);
    const long long r = i / g.nz;
    const int y = (int)(r % g.ny), x = (int)(r / g.ny);
    const long long p = ((long long)(x + AX) * g.py + (y + AY)) * g.pz + (z + AZ);
    const long long d = x * g.dstride[0] + y * g.dstride[1] + z * g.dstride[2];
    DBG_BOUNDS(p >= 0 && p < g.vol && d >= 0 && d < vol);
    dense[d] = round_scaled(acc[p], E);
  }
}

// ---------------------------------------------------------------------------------------
// LSQR over a ray set (include/sweeptt.h, sweeptt_rayset_lsqr; DESIGN §3.11)
// ---------------------------------------------------------------------------------------
// The vector passes of one LSQR iteration, every one float64 with DADD / DMUL only (no division or square root: the
// host forms the reciprocals and roots).  A pass that needs a norm squares its outputs and sums every block of
// LSQR_BLOCK consecutive squares with the halving tree a[i] = a[i] + a[i+h], h = 1024 .. 1 (elements past the end are
// +0); lsqr_reduce_kernel applies the same tree to the block sums until one value is left.  Which CTA takes which block
// changes nothing, so the sums are deterministic and independent of the grid.
constexpr int LSQR_THREADS = 256;
constexpr long long LSQR_BLOCK = 2048;

// Tree sum of block [base, base + 2048) of val(0 .. n-1); val(i) is called exactly once for every i < n of the block.
// s: 1024 doubles of shared memory.  Thread 0 returns the sum.
template <class F>
__device__ __forceinline__ double lsqr_block_sum(double* s, long long base, long long n, F&& val) {
  const int t = threadIdx.x;
#pragma unroll
  for (int k = 0; k < 1024 / LSQR_THREADS; ++k) {
    const int i = t + k * LSQR_THREADS;
    const double lo = base + i < n ? val(base + i) : 0.0;
    const double hi = base + i + 1024 < n ? val(base + i + 1024) : 0.0;
    s[i] = __dadd_rn(lo, hi);
  }
  __syncthreads();
  for (int h = 512; h >= 32; h >>= 1) {
    for (int i = t; i < h; i += LSQR_THREADS) s[i] = __dadd_rn(s[i], s[i + h]);
    __syncthreads();
  }
  double r = 0.0;
  if (t < 32) {
    r = s[t];
    for (int h = 16; h; h >>= 1) r = __dadd_rn(r, __shfl_down_sync(0xffffffffu, r, h));
  }
  __syncthreads();  // s is reused by the next block
  return r;
}

// First level: part[b] = tree sum of block b of val(0 .. n-1), the blocks shared out over the grid.
template <class F>
__device__ __forceinline__ void lsqr_blocks(long long n, double* part, F&& val) {
  __shared__ double s[1024];
  const long long nb = (n + LSQR_BLOCK - 1) / LSQR_BLOCK;
  for (long long b = blockIdx.x; b < nb; b += gridDim.x) {
    const double r = lsqr_block_sum(s, b * LSQR_BLOCK, n, val);
    if (threadIdx.x == 0) part[b] = r;
  }
}

// One CTA: the n block sums in part[] are summed level by level, in place (block b of a level is read before its sum
// goes to part[b], and b < LSQR_BLOCK * b' for every later block b'), until part[0] holds the total.
__global__ void __launch_bounds__(LSQR_THREADS) lsqr_reduce_kernel(double* part, long long n) {
  __shared__ double s[1024];
  while (n > 1) {
    const long long nb = (n + LSQR_BLOCK - 1) / LSQR_BLOCK;
    for (long long b = 0; b < nb; ++b) {
      const double r = lsqr_block_sum(s, b * LSQR_BLOCK, n, [&](long long i) { return part[i]; });
      if (threadIdx.x == 0) part[b] = r;
      __syncthreads();
    }
    n = nb;
  }
}

__device__ __forceinline__ double lsqr_sq(double a) { return __dmul_rn(a, a); }

// Row k of D (k < mD): fl(smooth * fl(v[n + e_a] - v[n])), the rows of axis 0, then 1, then 2, each in FLOATBOX order
// of the nodes n whose neighbour n + e_a is in the box.
__device__ __forceinline__ double lsqr_d_row(const LsqrArgs& a, long long k) {
  const long long nx = a.nx, ny = a.ny, nz = a.nz;
  const long long s0 = (nx - 1) * ny * nz, s1 = nx * (ny - 1) * nz;
  long long n, step;
  if (k < s0) {
    n = k;
    step = ny * nz;
  } else if ((k -= s0) < s1) {
    const long long z = k % nz, r = k / nz, y = r % (ny - 1), x = r / (ny - 1);
    n = (x * ny + y) * nz + z;
    step = nz;
  } else {
    k -= s1;
    n = k / (nz - 1) * nz + k % (nz - 1);
    step = 1;
  }
  DBG_BOUNDS(n >= 0 && n + step < nx * ny * nz);
  return __dmul_rn(a.smooth, __dsub_rn(a.v[n + step], a.v[n]));
}

// Component j of D^T y (y = the D rows of u): acc = +0; for a = 0, 1, 2: + y_a[j - e_a] if that node is in the box,
// then - y_a[j] if j + e_a is; fl(smooth * acc).
__device__ __forceinline__ double lsqr_dt(const LsqrArgs& a, long long j) {
  const long long nx = a.nx, ny = a.ny, nz = a.nz;
  const long long z = j % nz, r = j / nz, y = r % ny, x = r / ny;
  const double* u0 = a.u + a.m;
  const double* u1 = u0 + (nx - 1) * ny * nz;
  const double* u2 = u1 + nx * (ny - 1) * nz;
  double acc = 0.0;
  if (x > 0) acc = __dadd_rn(acc, u0[j - ny * nz]);
  if (x < nx - 1) acc = __dsub_rn(acc, u0[j]);
  const long long i1 = (x * (ny - 1) + y) * nz + z;  // row of node j along axis 1
  if (y > 0) acc = __dadd_rn(acc, u1[i1 - nz]);
  if (y < ny - 1) acc = __dsub_rn(acc, u1[i1]);
  const long long i2 = (x * ny + y) * (nz - 1) + z;  // ... along axis 2
  if (z > 0) acc = __dadd_rn(acc, u2[i2 - 1]);
  if (z < nz - 1) acc = __dsub_rn(acc, u2[i2]);
  return __dmul_rn(a.smooth, acc);
}

// Partials of sumsq(p[0 .. n)).
__global__ void __launch_bounds__(LSQR_THREADS) lsqr_sumsq_kernel(const double* __restrict__ p, long long n,
                                                                  double* __restrict__ part) {
  lsqr_blocks(n, part, [&](long long i) { return lsqr_sq(p[i]); });
}

// Pass A (first half): stage = float32(v), dense caller axes; launch_pad_box then pads it into the set's box.
__global__ void lsqr_to_f32_kernel(const double* __restrict__ v, float* __restrict__ stage, long long n) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    stage[i] = __double2float_rn(v[i]);
}

// Pass C: u = A v - alpha u, A v = [float64(io[row[i]]); D v], and the partials of sumsq(u).
__global__ void __launch_bounds__(LSQR_THREADS) lsqr_u_kernel(const LsqrArgs a, double alpha) {
  lsqr_blocks(a.m + a.mD, a.part, [&](long long i) {
    const double av = i < a.m ? (double)a.io[a.row[i]] : lsqr_d_row(a, i - a.m);
    const double u = __dsub_rn(av, __dmul_rn(alpha, a.u[i]));
    a.u[i] = u;
    return lsqr_sq(u);
  });
}

// Pass D: u = inv_beta * u; the G rows, as float32 weights W, go to io[row[i]] (zeroed by the caller), and the bits of
// max |W| to *wmax (non-negative floats order like their bits).
__global__ void __launch_bounds__(LSQR_THREADS) lsqr_scale_u_kernel(const LsqrArgs a, double inv_beta) {
  unsigned mx = 0;
  const long long n = a.m + a.mD;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const double u = __dmul_rn(inv_beta, a.u[i]);
    a.u[i] = u;
    if (i < a.m) {
      const float W = __double2float_rn(u);
      a.io[a.row[i]] = W;
      mx = max(mx, __float_as_uint(W) & 0x7fffffffu);
    }
  }
  for (int o = 16; o; o >>= 1) mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  if ((threadIdx.x & 31) == 0 && mx) atomicMax(a.wmax, mx);
}

// Pass F: v = A^T u - beta v, A^T u = fl(float64(grad) + D^T u_D) (the D term only with smoothing; grad = the set's
// rounded back-projection in stage), and the partials of sumsq(v).
__global__ void __launch_bounds__(LSQR_THREADS) lsqr_v_kernel(const LsqrArgs a, double beta) {
  lsqr_blocks((long long)a.nx * a.ny * a.nz, a.part, [&](long long j) {
    double g = (double)a.stage[j];
    if (a.smooth > 0.0) g = __dadd_rn(g, lsqr_dt(a, j));
    const double v = __dsub_rn(g, __dmul_rn(beta, a.v[j]));
    a.v[j] = v;
    return lsqr_sq(v);
  });
}

__global__ void lsqr_scale_kernel(double* __restrict__ p, long long n, double s) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    p[i] = __dmul_rn(s, p[i]);
}

// Step 7: dk = inv_rho * w (only its sumsq partials are kept), x = x + t1 w, w = v + t2 w.
__global__ void __launch_bounds__(LSQR_THREADS) lsqr_xw_kernel(const LsqrArgs a, double t1, double t2, double inv_rho) {
  lsqr_blocks((long long)a.nx * a.ny * a.nz, a.part, [&](long long j) {
    const double w = a.w[j];
    const double dk = __dmul_rn(inv_rho, w);
    a.x[j] = __dadd_rn(a.x[j], __dmul_rn(t1, w));
    a.w[j] = __dadd_rn(a.v[j], __dmul_rn(t2, w));
    return lsqr_sq(dk);
  });
}

// ---------------------------------------------------------------------------------------
// event location (include/sweeptt.h, sweeptt_locate_events / sweeptt_misfit_box; DESIGN §3.10)
// ---------------------------------------------------------------------------------------
constexpr int LOC_THREADS = 512;
constexpr unsigned LOC_EXCLUDED = 0x7f800001u;  // key bits of an excluded node: after every float32 misfit, +INF too

// RN(a / k) for a finite double a and an integer 1 <= k < 2^26, with DMUL / DADD only: ptxas expands div.rn.f64 into
// a DFMA sequence, and these kernels keep no fused multiply-add.  q = RN(a * rk), rk = RN(1/k), is within two ulps of
// a/k.  The remainder a - q*k is exact: q splits (Veltkamp, 2^27 + 1) into a 26-bit qh and a 27-bit ql, so qh*k and
// ql*k are exact, a - qh*k is exact by Sterbenz's lemma, and the last difference is a multiple of ulp(q) below
// 2^53 ulp(q).  Its sign tells on which side of q the quotient lies; q steps to that neighbour while the neighbour is
// nearer.  a/k is never halfway between two doubles (an odd multiple of a 54-bit odd significand needs more than 53
// bits), so the nearer of two neighbours is RN(a/k).
__device__ __forceinline__ double loc_remainder(double a, double q, double k) {
  const double c = __dmul_rn(134217729.0, q);
  const double qh = __dsub_rn(c, __dsub_rn(c, q));
  const double ql = __dsub_rn(q, qh);
  return __dsub_rn(__dsub_rn(a, __dmul_rn(qh, k)), __dmul_rn(ql, k));
}
__device__ __forceinline__ double loc_div(double a, int k, double rk) {
  if (k == 0) return __longlong_as_double(0x7ff8000000000000ll);  // 0 / 0
  const double kd = (double)k;
  double q = __dmul_rn(a, rk);
  double r = loc_remainder(a, q, kd);
  for (int it = 0; it < 4 && r != 0.0; ++it) {
    // the neighbour of q towards a/k: a larger magnitude when r has q's sign
    const long long step = ((r > 0.0) == (q > 0.0)) ? 1 : -1;
    const double qn = __longlong_as_double(__double_as_longlong(q) + step);
    const double rn = loc_remainder(a, qn, kd);
    if (!(fabs(rn) < fabs(r))) break;
    q = qn;
    r = rn;
  }
  return q;
}

// The per-node formula of include/sweeptt.h, at NB nodes of one event: the ONE implementation, shared by locate_kernel,
// misfit_box_kernel and locate_finish_kernel.  tt(s, q) is station s's travel time at node q as a double; ps / po are
// the event's k picks, ascending.  bits[q] = float bits of the misfit, or LOC_EXCLUDED; t0[q] = the origin time.
template <int NB, class TT>
__device__ __forceinline__ void event_misfit(const int* __restrict__ ps, const double* __restrict__ po, int k, double rk,
                                             const TT& tt, unsigned (&bits)[NB], double (&t0)[NB]) {
  double acc[NB], m[NB];
#pragma unroll
  for (int q = 0; q < NB; ++q) acc[q] = 0.0, m[q] = 0.0;
#pragma unroll 4
  for (int j = 0; j < k; ++j) {
    const int s = ps[j];
    const double o = po[j];
#pragma unroll
    for (int q = 0; q < NB; ++q) acc[q] = __dadd_rn(acc[q], __dsub_rn(o, tt(s, q)));
  }
#pragma unroll
  for (int q = 0; q < NB; ++q) t0[q] = loc_div(acc[q], k, rk);
#pragma unroll 4
  for (int j = 0; j < k; ++j) {
    const int s = ps[j];
    const double o = po[j];
#pragma unroll
    for (int q = 0; q < NB; ++q) {
      const double u = __dsub_rn(__dsub_rn(o, tt(s, q)), t0[q]);
      m[q] = __dadd_rn(m[q], __dmul_rn(u, u));
    }
  }
#pragma unroll
  for (int q = 0; q < NB; ++q) {
    // picks are finite, so a +INF time makes acc -INF or NaN; a finite acc rules every +INF out
    bool excluded = false;
    if (!isfinite(acc[q]))
      for (int j = 0; j < k; ++j) excluded |= tt(ps[j], q) == CUDART_INF;
    bits[q] = excluded ? LOC_EXCLUDED : __float_as_uint(__double2float_rn(m[q]));
  }
}

struct LocSmemTT {  // the CTA's staged times: station s, node q of this lane at base[s * B + 32 * q]
  const double* base;
  int B;
  __device__ __forceinline__ double operator()(int s, int q) const { return base[s * B + 32 * q]; }
};
struct LocBoxTT {   // the padded boxes in global memory, at one node
  const float* tt;
  long long vol, p;
  __device__ __forceinline__ double operator()(int s, int) const { return (double)__ldg(tt + s * vol + p); }
};

// Caller FLOATBOX index and padded index of kernel-order node i = (x*ny + y)*nz + z.
__device__ __forceinline__ void loc_node(const BoxGeom& g, long long i, long long* p, long long* d) {
  const int z = (int)(i % g.nz);
  const long long r = i / g.nz;
  const int y = (int)(r % g.ny), x = (int)(r / g.ny);
  *p = ((long long)(x + AX) * g.py + (y + AY)) * g.pz + (z + AZ);
  *d = x * g.dstride[0] + y * g.dstride[1] + z * g.dstride[2];
}

// A CTA owns B = 32*NB consecutive nodes in kernel order (a run along kernel z: coalesced reads), stages the times of
// every station there once (doubles, [nsta][B]), then its warps take the launch's events in turn: lane l evaluates
// nodes l, l+32, ... of the run for the warp's event, whose picks are warp-uniform loads.  The warp's smallest key goes
// to the event with one 64-bit atomicMin (integer min: the result does not depend on the schedule).
template <int NB>
__global__ void __launch_bounds__(LOC_THREADS, 1) locate_kernel(const LocateArgs a) {
  constexpr int B = 32 * NB;
  extern __shared__ double s_tt[];
  __shared__ long long s_p[B];
  __shared__ unsigned s_j[B];
  const long long D = (long long)a.g.nx * a.g.ny * a.g.nz;
  const long long n0 = (long long)blockIdx.x * B;
  for (int b = threadIdx.x; b < B; b += blockDim.x) {
    long long p = -1, d = 0;
    if (n0 + b < D) loc_node(a.g, n0 + b, &p, &d);
    s_p[b] = p;
    s_j[b] = (unsigned)d;
  }
  __syncthreads();
  for (int idx = threadIdx.x; idx < a.nsta * B; idx += blockDim.x) {
    const int s = idx / B, b = idx % B;
    const long long p = s_p[b];
    s_tt[idx] = p >= 0 ? (double)__ldg(a.tt + s * a.g.vol + p) : CUDART_INF;
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  bool live[NB];
  unsigned jn[NB];
#pragma unroll
  for (int q = 0; q < NB; ++q) live[q] = s_p[32 * q + lane] >= 0, jn[q] = s_j[32 * q + lane];
  const LocSmemTT tt{s_tt + lane, B};
  for (int e = a.e_begin + warp; e < a.e_begin + a.e_count; e += LOC_THREADS / 32) {
    const int off = a.pick_off[e], k = a.pick_off[e + 1] - off;
    if (k == 0) continue;
    unsigned bits[NB];
    double t0[NB];
    event_misfit<NB>(a.pick_sta + off, a.pick_obs + off, k, a.pick_rk[e], tt, bits, t0);
    unsigned long long best = ~0ull;
#pragma unroll
    for (int q = 0; q < NB; ++q)
      if (live[q]) best = min(best, ((unsigned long long)bits[q] << 32) | jn[q]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) best = min(best, __shfl_xor_sync(0xffffffffu, best, o));
    if (lane == 0 && best != ~0ull) atomicMin(a.key + e, best);
  }
}

__global__ void locate_finish_kernel(const LocateArgs a, int nev) {
  const BoxGeom& g = a.g;
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < nev; e += gridDim.x * blockDim.x) {
    const int off = a.pick_off[e], k = a.pick_off[e + 1] - off;
    const unsigned long long key = a.key[e];
    a.npicks[e] = k;
    if (k == 0 || (unsigned)(key >> 32) == LOC_EXCLUDED || key == ~0ull) {
      a.node[3 * e] = a.node[3 * e + 1] = a.node[3 * e + 2] = -1;
      a.misfit[e] = CUDART_INF_F;
      a.origin[e] = __longlong_as_double(0x7ff8000000000000ll);
      a.status[e] = k == 0 ? SWEEPTT_LOC_NO_PICKS : SWEEPTT_LOC_UNREACHED;
      continue;
    }
    // caller coordinates of j = (c0*n1 + c1)*n2 + c2, then kernel axes (kernel axis q = caller axis perm[q])
    int n[3], c[3];
    n[g.perm[0]] = g.nx; n[g.perm[1]] = g.ny; n[g.perm[2]] = g.nz;
    const unsigned long long j = key & 0xffffffffull;
    c[2] = (int)(j % n[2]);
    c[1] = (int)(j / n[2] % n[1]);
    c[0] = (int)(j / n[2] / n[1]);
    const long long p = ((long long)(c[g.perm[0]] + AX) * g.py + (c[g.perm[1]] + AY)) * g.pz + (c[g.perm[2]] + AZ);
    unsigned bits[1];
    double t0[1];
    event_misfit<1>(a.pick_sta + off, a.pick_obs + off, k, a.pick_rk[e], LocBoxTT{a.tt, g.vol, p}, bits, t0);
    a.node[3 * e] = c[0]; a.node[3 * e + 1] = c[1]; a.node[3 * e + 2] = c[2];
    a.misfit[e] = __uint_as_float(bits[0]);
    a.origin[e] = t0[0];
    a.status[e] = SWEEPTT_LOC_OK;
  }
}

__global__ void __launch_bounds__(256) misfit_box_kernel(const LocateArgs a, float* __restrict__ dense) {
  const long long D = (long long)a.g.nx * a.g.ny * a.g.nz;
  const int k = a.pick_off[1] - a.pick_off[0];
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < D; i += (long long)gridDim.x * blockDim.x) {
    long long p, d;
    loc_node(a.g, i, &p, &d);
    unsigned bits[1];
    double t0[1];
    event_misfit<1>(a.pick_sta, a.pick_obs, k, a.pick_rk[0], LocBoxTT{a.tt, a.g.vol, p}, bits, t0);
    dense[d] = bits[0] == LOC_EXCLUDED ? CUDART_INF_F : __uint_as_float(bits[0]);
  }
}

// ---------------------------------------------------------------------------------------
// float-box utilities
// ---------------------------------------------------------------------------------------
__global__ void fill_kernel(float4* p, long long n4, float value) {
  const float4 v = make_float4(value, value, value, value);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x)
    p[i] = v;
}
__global__ void fill_u32_kernel(unsigned* p, long long n, unsigned value) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    p[i] = value;
}
__global__ void pad_kernel(const float* __restrict__ dense, float* __restrict__ padded, BoxGeom g) {
  const long long vol = (long long)g.nx * g.ny * g.nz;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < vol; i += (long long)gridDim.x * blockDim.x) {
    const int z = (int)(i % g.nz);
    const long long r = i / g.nz;
    const int y = (int)(r % g.ny), x = (int)(r / g.ny);
    padded[((long long)(x + AX) * g.py + (y + AY)) * g.pz + (z + AZ)] =
        dense[x * g.dstride[0] + y * g.dstride[1] + z * g.dstride[2]];
  }
}
__global__ void unpad_kernel(const float* __restrict__ padded, float* __restrict__ dense, BoxGeom g) {
  const long long vol = (long long)g.nx * g.ny * g.nz;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < vol; i += (long long)gridDim.x * blockDim.x) {
    const int z = (int)(i % g.nz);
    const long long r = i / g.nz;
    const int y = (int)(r % g.ny), x = (int)(r / g.ny);
    dense[x * g.dstride[0] + y * g.dstride[1] + z * g.dstride[2]] =
        padded[((long long)(x + AX) * g.py + (y + AY)) * g.pz + (z + AZ)];
  }
}
// Statistics of the model in one pass over the dense staged box: out[0] = float bits of the smallest slowness,
// out[1] != 0 when a value is negative or NaN (switches the downwind filter off), then (8-byte aligned) the sum
// (double) and the count (unsigned long long) of the finite values -- the mean only scales the activation bucket --
// then out[6] = bits of the largest finite slowness and out[7] = bits of the smallest positive one (+INF if none).
// The bits of non-negative floats order like the floats; -0.0 counts as +0.0 (its bits would order above +INF).
__global__ void min_slowness_kernel(const float* __restrict__ dense, long long n, unsigned* out) {
  unsigned m = 0x7f800000u, bad = 0u, mx = 0u, pos = 0x7f800000u;
  double sum = 0.0;
  unsigned long long cnt = 0ull;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float v = dense[i];
    if (v >= 0.f) {
      const unsigned b = __float_as_uint(v) & 0x7fffffffu;
      m = min(m, b);
      if (b != 0x7f800000u) mx = max(mx, b);
      if (b != 0u) pos = min(pos, b);
    } else {
      bad = 1u;
    }
    if (v == v && fabsf(v) != CUDART_INF_F) { sum += (double)v; ++cnt; }
  }
  m = __reduce_min_sync(0xffffffffu, m);
  bad = __reduce_or_sync(0xffffffffu, bad);
  mx = __reduce_max_sync(0xffffffffu, mx);
  pos = __reduce_min_sync(0xffffffffu, pos);
  for (int o = 16; o; o >>= 1) {
    sum += __shfl_xor_sync(0xffffffffu, sum, o);
    cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
  }
  if ((threadIdx.x & 31) == 0) {
    atomicMin(&out[0], m);
    if (bad) atomicOr(&out[1], 1u);
    atomicAdd(reinterpret_cast<double*>(out + 2), sum);
    atomicAdd(reinterpret_cast<unsigned long long*>(out + 4), cnt);
    atomicMax(&out[6], mx);
    atomicMin(&out[7], pos);
  }
}
cudaError_t launch_min_slowness(const float* dense, long long n, unsigned* out8, cudaStream_t stream) {
  static const unsigned init[8] = {0x7f800000u, 0u, 0u, 0u, 0u, 0u, 0u, 0x7f800000u};
  cudaError_t e = cudaMemcpyAsync(out8, init, sizeof init, cudaMemcpyHostToDevice, stream);  // (pageable source: staged at call time)
  if (e != cudaSuccess) return e;
  min_slowness_kernel<<<1184, 256, 0, stream>>>(dense, n, out8);
  return cudaGetLastError();
}

// one block per source: tt[start] = 0 and every tile within star reach of the start's tile goes on list 0
__global__ void init_sources_kernel(const RelaxArgs a) {
  const int s = blockIdx.x;
  const int px = a.src_xyz[3 * s], py = a.src_xyz[3 * s + 1], pz = a.src_xyz[3 * s + 2];
  if (px < 0 || px >= a.g.nx || py < 0 || py >= a.g.ny || pz < 0 || pz >= a.g.nz) return;
  // (one grid over several devices: the owner of the start's x block writes the 0, every part lists its own tiles)
  if (threadIdx.x == 63 && (a.nparts <= 1 || a.tx_owner[px / TX] == a.part))
    a.tt[(size_t)s * a.g.vol + ((size_t)(px + AX) * a.g.py + (py + AY)) * a.g.pz + (pz + AZ)] = 0.0f;
  if (threadIdx.x < NMARK) {
    const int tid = threadIdx.x;
    const int ux = px / TX + tid / 9 - XREACH, uy = py / TY + (tid / 3) % 3 - 1, uz = pz / TZ + tid % 3 - 1;
    if (ux >= 0 && ux < a.g.ntx && uy >= 0 && uy < a.g.nty && uz >= 0 && uz < a.g.ntz &&
        (a.nparts <= 1 || a.tx_owner[ux] == a.part)) {
      const unsigned ntiles = a.g.ntx * a.g.nty * a.g.ntz;
      const unsigned pos = atomicAdd(&a.st->count[0], 1u);
      a.worklist[pos] = s * ntiles + (ux * a.g.nty + uy) * a.g.ntz + uz;
    }
  }
}

// ---------------------------------------------------------------------------------------
// launchers
// ---------------------------------------------------------------------------------------
int tiled_variant_for_radius(int r) {
  if (r <= 2) return 2;
  if (r <= 4) return 4;
  if (r <= 7) return 7;
  return 0;
}
void tiled_variant_dims(int rxy, int* sxd, int* syd, int* szd) {
  *sxd = TX + 2 * rxy; *syd = TY + 2 * rxy; *szd = SZD;
}

// stock stars: pattern lists generated from the reference's shipped star files
#define SWEEPTT_STOCK_STAR(id, name, rxy, ...) using Star_##name = MaskList<__VA_ARGS__>;
#include "stock_stars.inc"
#undef SWEEPTT_STOCK_STAR
using StarGeneric = MaskList<>;

template <uint32_t... M>
static int masks_match(MaskList<M...>, const uint32_t* masks, int n) {
  constexpr uint32_t want[] = {M..., 0u};
  if (n != (int)sizeof...(M)) return 0;
  for (int i = 0; i < n; ++i)
    if (masks[i] != want[i]) return 0;
  return 1;
}

int tiled_stock_star_for(const uint32_t* masks_ascending, int n, int rxy_needed) {
#define SWEEPTT_STOCK_STAR(id, name, rxy, ...) \
  if (rxy_needed == rxy && masks_match(Star_##name{}, masks_ascending, n)) return id;
#include "stock_stars.inc"
#undef SWEEPTT_STOCK_STAR
  return 0;
}

// compute warps per CTA: the 3-FS star has too few columns to share out 16 ways; its small staged boxes
// let three 5-warp CTAs share an SM instead
template <int RXY>
constexpr int warps_for() { return RXY == 2 ? 4 : MAX_WARPS; }

template <int RXY, typename STAR>
static cudaError_t prepare_variant(int device, TiledLaunch* out) {
  using D = TileDims<RXY>;
  constexpr int NW = warps_for<RXY>();
  const size_t smem = D::SMEM;
  cudaError_t e = cudaFuncSetAttribute(relax_tiled<RXY, STAR, NW, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  e = cudaFuncSetAttribute(relax_tiled<RXY, STAR, NW, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  int per_sm = 0, per_sm_p = 0, sms = 0;
  e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, relax_tiled<RXY, STAR, NW, false>, 32 * NW, smem);
  if (e != cudaSuccess) return e;
  e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm_p, relax_tiled<RXY, STAR, NW, true>, 32 * NW, smem);
  if (e != cudaSuccess) return e;
  e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
  if (e != cudaSuccess) return e;
  if (per_sm < 1 || per_sm_p < 1) return cudaErrorLaunchOutOfResources;
  out->rxy = RXY;
  out->grid = per_sm * sms;
  out->grid_persistent = per_sm_p * sms;
  out->smem_bytes = smem;
  out->nw = NW;
  return cudaSuccess;
}
template <int RXY, typename STAR>
static void launch_variant(const TiledLaunch& tl, const CUtensorMap& tm_slow, const CUtensorMap& tm_tt,
                           const RelaxArgs& a, bool persistent, cudaStream_t stream) {
  constexpr int NW = warps_for<RXY>();
  if (persistent)
    relax_tiled<RXY, STAR, NW, true><<<tl.grid_persistent, dim3(32, NW, 1), tl.smem_bytes, stream>>>(tm_slow, tm_tt, a);
  else
    relax_tiled<RXY, STAR, NW, false><<<tl.grid, dim3(32, NW, 1), tl.smem_bytes, stream>>>(tm_slow, tm_tt, a);
}
__global__ void compact_fused(const RelaxArgs a, unsigned long long cond);
cudaError_t tiled_prepare(int rxy, int stock_id, int device, TiledLaunch* out) {
  out->stock_id = stock_id;
  {  // the single-block compaction keeps its keys in (opt-in) dynamic shared memory; per device
    cudaError_t e = cudaFuncSetAttribute(compact_fused, cudaFuncAttributeMaxDynamicSharedMemorySize, 49152 * 4);
    if (e != cudaSuccess) return e;
  }
#define SWEEPTT_STOCK_STAR(id, name, r, ...) \
  if (stock_id == id) return prepare_variant<r, Star_##name>(device, out);
#include "stock_stars.inc"
#undef SWEEPTT_STOCK_STAR
  switch (rxy) {
    case 2: return prepare_variant<2, StarGeneric>(device, out);
    case 4: return prepare_variant<4, StarGeneric>(device, out);
    case 7: return prepare_variant<7, StarGeneric>(device, out);
  }
  return cudaErrorInvalidValue;
}

static cudaError_t launch_relax_any(const TiledLaunch& tl, const CUtensorMap& tm_slow, const CUtensorMap& tm_tt,
                                    const RelaxArgs& a, bool persistent, cudaStream_t stream) {
#define SWEEPTT_STOCK_STAR(id, name, r, ...)                                   \
  if (tl.stock_id == id) {                                                     \
    launch_variant<r, Star_##name>(tl, tm_slow, tm_tt, a, persistent, stream); \
    return cudaGetLastError();                                                 \
  }
#include "stock_stars.inc"
#undef SWEEPTT_STOCK_STAR
  switch (tl.rxy) {
    case 2: launch_variant<2, StarGeneric>(tl, tm_slow, tm_tt, a, persistent, stream); break;
    case 4: launch_variant<4, StarGeneric>(tl, tm_slow, tm_tt, a, persistent, stream); break;
    case 7: launch_variant<7, StarGeneric>(tl, tm_slow, tm_tt, a, persistent, stream); break;
    default: return cudaErrorInvalidValue;
  }
  return cudaGetLastError();
}
cudaError_t launch_relax_tiled(const TiledLaunch& tl, const CUtensorMap& tm_slow, const CUtensorMap& tm_tt,
                               const RelaxArgs& a, cudaStream_t stream) {
  return launch_relax_any(tl, tm_slow, tm_tt, a, false, stream);
}
cudaError_t launch_relax_persistent(const TiledLaunch& tl, const CUtensorMap& tm_slow, const CUtensorMap& tm_tt,
                                    const RelaxArgs& a, cudaStream_t stream) {
  return launch_relax_any(tl, tm_slow, tm_tt, a, true, stream);
}
// after a single-launch solve: fold every key that is still pending into kmin_bits (must stay INF)
cudaError_t launch_persist_check(const RelaxArgs& a, cudaStream_t stream) {
  const size_t total = (size_t)a.nsrc * a.g.ntx * a.g.nty * a.g.ntz;
  scan_min_key<<<(unsigned)std::min<size_t>(296, (total + 255) / 256), 256, 0, stream>>>(a);
  return cudaGetLastError();
}
size_t tiled_persistent_max_keys(int rxy) {  // the generation builder caches every key in the idle TMA ring
  switch (rxy) {
    case 2: return 4 * (size_t)TileDims<2>::BOX_STRIDE;
    case 4: return 4 * (size_t)TileDims<4>::BOX_STRIDE;
    case 7: return 4 * (size_t)TileDims<7>::BOX_STRIDE;
  }
  return 0;
}
// generation 0 = the list init_sources_kernel wrote: book its tiles as busy / in flight
__global__ void persist_begin_kernel(const RelaxArgs a) {
  SolveState* S = a.st;
  const unsigned cnt = S->count[0];
  for (unsigned i = threadIdx.x; i < cnt; i += blockDim.x) a.busy[a.worklist[i]] = 1u;
  if (threadIdx.x == 0) {
    S->gen = 0u; S->builder = 0u; S->done = 0u;
    S->inflight = cnt;
    S->gslot[0] = (unsigned long long)cnt << 32;
  }
}
cudaError_t launch_persist_begin(const RelaxArgs& a, cudaStream_t stream) {
  const size_t total = (size_t)a.nsrc * a.g.ntx * a.g.nty * a.g.ntz;
  cudaError_t e = cudaMemsetAsync(a.busy, 0, total * sizeof(unsigned), stream);
  if (e != cudaSuccess) return e;
  persist_begin_kernel<<<1, 256, 0, stream>>>(a);
  return cudaGetLastError();
}

// Small problems (<= 64 Ki tiles): ONE block does the min-scan, the selection AND orders the
// selected tiles by activation key (counting sort into 32 key bins), so the persistent relaxation
// CTAs pop tiles in increasing travel-time order -- later tiles of a round then read what earlier
// ones produced (Gauss-Seidel along the propagation direction) -- and a round is one launch shorter.
constexpr int FUSED_MAX_KEYS = 49152;  // cached in shared memory (192 KB)
constexpr int FUSED_BINS = 32;
__global__ void __launch_bounds__(1024) compact_fused(const RelaxArgs a, unsigned long long cond) {
  extern __shared__ unsigned s_keys[];  // the keys are read from global memory ONCE; the three passes run on this copy
  __shared__ unsigned s_min;
  __shared__ unsigned s_bin[FUSED_BINS + 1];
  SolveState* S = a.st;
  const int nxt = S->parity ^ 1;
  const unsigned total = (unsigned)((size_t)a.nsrc * a.g.ntx * a.g.nty * a.g.ntz);
  if (threadIdx.x == 0) s_min = 0x7f800000u;
  if (threadIdx.x <= FUSED_BINS) s_bin[threadIdx.x] = 0;
  __syncthreads();
  unsigned m = 0x7f800000u;
#pragma unroll 8
  for (unsigned i = threadIdx.x; i < total; i += 1024) {
    const unsigned k = a.key[i];
    s_keys[i] = k;
    m = min(m, k);
  }
  m = __reduce_min_sync(0xffffffffu, m);
  if ((threadIdx.x & 31) == 0 && m != 0x7f800000u) atomicMin(&s_min, m);
  __syncthreads();
  if (a.nparts > 1) {  // (see select_tiles)
    if (threadIdx.x == 0) {
      unsigned g = s_min;
      const unsigned own = g;
      st_volatile_u32(a.part_kmin[a.part], g);
      for (int q = 0; q < a.nparts; ++q)
        if (q != a.part) g = min(g, ld_volatile_u32(a.part_kmin[q]));
      if (own != 0x7f800000u) g = max(g, __float_as_uint(fmaxf(0.f, __uint_as_float(own) - a.front_slack)));
      s_min = g;
    }
    __syncthreads();
  }
  const float kmin = __uint_as_float(s_min);
  const bool all = a.bucket < 0.f;
  const unsigned thr = all ? 0x7f7fffffu : __float_as_uint(kmin + a.bucket);
  const float scale = a.bin_scale;  // FUSED_BINS / bucket, divided on the host
  // pass A: histogram of the selected tiles' key bins
  for (unsigned i = threadIdx.x; i < total; i += 1024) {
    const unsigned k = s_keys[i];
    if (k != 0x7f800000u && k <= thr) {
      const int b = min(FUSED_BINS - 1, (int)((__uint_as_float(k) - kmin) * scale));
      atomicAdd(&s_bin[b + 1], 1u);
    }
  }
  __syncthreads();
  if (threadIdx.x == 0)
    for (int b = 0; b < FUSED_BINS; ++b) s_bin[b + 1] += s_bin[b];  // exclusive starts in s_bin[0..BINS-1]
  __syncthreads();
  const unsigned cnt = s_bin[FUSED_BINS];
  __syncthreads();
  // pass B: scatter in bin order, clear the keys
  unsigned* wl = a.worklist + (size_t)nxt * a.cap;
  for (unsigned i = threadIdx.x; i < total; i += 1024) {
    const unsigned k = s_keys[i];
    if (k != 0x7f800000u && k <= thr) {
      const int b = min(FUSED_BINS - 1, (int)((__uint_as_float(k) - kmin) * scale));
      wl[atomicAdd(&s_bin[b], 1u)] = i;
      a.key[i] = 0x7f800000u;
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    S->cursor = 0;
    S->count[nxt] = cnt;
    S->count[nxt ^ 1] = 0;
    S->parity = nxt;
    S->round += 1;
    S->kmin_bits = 0x7f800000u;
#if __CUDA_ARCH__ >= 900
    if (cond) {
      const bool more = (cnt != 0) && (S->max_rounds == 0 || S->round < S->max_rounds);
      cudaGraphSetConditional((cudaGraphConditionalHandle)cond, more ? 1u : 0u);
    }
#endif
  }
}

cudaError_t launch_compact(const RelaxArgs& a, unsigned long long cond, cudaStream_t stream) {
  const size_t total = (size_t)a.nsrc * a.g.ntx * a.g.nty * a.g.ntz;
  if (total <= (size_t)FUSED_MAX_KEYS) {
    compact_fused<<<1, 1024, (total * 4 + 15) / 16 * 16, stream>>>(a, cond);
    return cudaGetLastError();
  }
  const unsigned blocks = (unsigned)((total + 255) / 256);
  scan_min_key<<<std::min(blocks, 1184u), 256, 0, stream>>>(a);
  select_tiles<<<blocks, 256, 0, stream>>>(a, cond);
  return cudaGetLastError();
}

cudaError_t launch_relax_simple(const RelaxArgs& a, const StarDev* star, int nstar,
                                unsigned long long pulls_per_round, cudaStream_t stream) {
  dim3 grid(a.g.nx * a.g.ny, (a.g.nz + 127) / 128, a.nsrc);
  relax_simple<<<grid, 128, 0, stream>>>(a, star, nstar, pulls_per_round);
  return cudaGetLastError();
}
cudaError_t launch_advance_simple(SolveState* st, unsigned long long cond, cudaStream_t stream) {
  advance_simple<<<1, 1, 0, stream>>>(st, cond);
  return cudaGetLastError();
}

cudaError_t launch_count_violations(const RelaxArgs& a, int source, const StarDev* star, int nstar,
                                    unsigned long long* out, cudaStream_t stream) {
  dim3 grid(a.g.nx * a.g.ny, (a.g.nz + 127) / 128, 1);
  count_violations_kernel<<<grid, 128, 0, stream>>>(a, source, star, nstar, out);
  return cudaGetLastError();
}

size_t trace_rays_smem_bytes(int npull) { return (size_t)npull * sizeof(RayPull); }

cudaError_t launch_trace_rays(const TraceArgs& t, int device, cudaStream_t stream) {
  static_assert(sizeof(RayPull) == 16, "one LDS.128 per pull entry");
  const size_t smem = trace_rays_smem_bytes(t.npull);
  cudaError_t e = cudaFuncSetAttribute(trace_rays_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  int sms = 0, per_sm = 0;
  e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
  if (e != cudaSuccess) return e;
  e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, trace_rays_kernel, TRACE_THREADS, smem);
  if (e != cudaSuccess) return e;
  if (per_sm < 1) return cudaErrorInvalidConfiguration;
  const long long need = (t.nrays + TRACE_THREADS / 32 - 1) / (TRACE_THREADS / 32);
  const int grid = (int)std::max(1LL, std::min<long long>(need, (long long)sms * per_sm));
  trace_rays_kernel<<<grid, TRACE_THREADS, smem, stream>>>(t);
  return cudaGetLastError();
}

cudaError_t ray_walk_prepare(bool backproject, int npull, int max_nodes, long long nrays, int device, RayWalkLaunch* out) {
  const void* fn = backproject ? (const void*)ray_backproject_kernel : (const void*)ray_project_kernel;
  const size_t table = (size_t)npull * sizeof(RayPull);
  const size_t with_path = table + (size_t)(TRACE_THREADS / 32) * max_nodes * sizeof(unsigned short);
  int sms = 0, optin = 0, per_sm_table = 0, per_sm_path = 0;
  cudaError_t e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
  if (e != cudaSuccess) return e;
  e = cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device);
  if (e != cudaSuccess) return e;
  const bool fits = with_path <= (size_t)optin;
  e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(fits ? with_path : table));
  if (e != cudaSuccess) return e;
  e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm_table, fn, TRACE_THREADS, table);
  if (e != cudaSuccess) return e;
  if (fits) {
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm_path, fn, TRACE_THREADS, with_path);
    if (e != cudaSuccess) return e;
  }
  out->path_in_smem = fits && per_sm_path == per_sm_table;
  const int per_sm = out->path_in_smem ? per_sm_path : per_sm_table;
  if (per_sm < 1) return cudaErrorInvalidConfiguration;
  out->smem = out->path_in_smem ? with_path : table;
  const long long need = (nrays + TRACE_THREADS / 32 - 1) / (TRACE_THREADS / 32);
  out->grid = (int)std::max(1LL, std::min<long long>(need, (long long)sms * per_sm));
  out->path_entries = out->path_in_smem ? 0 : (long long)out->grid * (TRACE_THREADS / 32) * max_nodes;
  return cudaSuccess;
}

cudaError_t launch_ray_walk(bool backproject, const RayWalkLaunch& l, const TomoArgs& a, cudaStream_t stream) {
  if (backproject)
    ray_backproject_kernel<<<l.grid, TRACE_THREADS, l.smem, stream>>>(a);
  else
    ray_project_kernel<<<l.grid, TRACE_THREADS, l.smem, stream>>>(a);
  return cudaGetLastError();
}

// Persistent warp-per-ray grid with the pull table in shared memory (the ray-set kernels).
static cudaError_t rayset_grid(const void* fn, int npull, long long nrays, int device, int* grid, size_t* smem) {
  *smem = (size_t)npull * sizeof(RayPull);
  cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)*smem);
  if (e != cudaSuccess) return e;
  int sms = 0, per_sm = 0;
  e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
  if (e != cudaSuccess) return e;
  e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, TRACE_THREADS, *smem);
  if (e != cudaSuccess) return e;
  if (per_sm < 1) return cudaErrorInvalidConfiguration;
  const long long need = (nrays + TRACE_THREADS / 32 - 1) / (TRACE_THREADS / 32);
  *grid = (int)std::max(1LL, std::min<long long>(need, (long long)sms * per_sm));
  return cudaSuccess;
}

cudaError_t launch_rayset_record(const TomoArgs& a, int device, cudaStream_t stream) {
  int grid;
  size_t smem;
  cudaError_t e = rayset_grid((const void*)rayset_record_kernel, a.t.npull, a.t.nrays, device, &grid, &smem);
  if (e != cudaSuccess) return e;
  rayset_record_kernel<<<grid, TRACE_THREADS, smem, stream>>>(a);
  return cudaGetLastError();
}

cudaError_t launch_rayset_compact(const unsigned short* staging, int max_nodes, const long long* off, long long nrays,
                                  unsigned short* dst, cudaStream_t stream) {
  const long long need = (nrays + TRACE_THREADS / 32 - 1) / (TRACE_THREADS / 32);
  rayset_compact_kernel<<<(unsigned)std::min<long long>(need, 4096), TRACE_THREADS, 0, stream>>>(staging, max_nodes, off,
                                                                                                 nrays, dst);
  return cudaGetLastError();
}

cudaError_t launch_rayset_walk(bool backproject, const RaySetArgs& s, int device, cudaStream_t stream) {
  const void* fn = backproject ? (const void*)rayset_backproject_kernel : (const void*)rayset_project_kernel;
  int grid;
  size_t smem;
  cudaError_t e = rayset_grid(fn, s.a.t.npull, s.a.t.nrays, device, &grid, &smem);
  if (e != cudaSuccess) return e;
  if (backproject)
    rayset_backproject_kernel<<<grid, TRACE_THREADS, smem, stream>>>(s);
  else
    rayset_project_kernel<<<grid, TRACE_THREADS, smem, stream>>>(s);
  return cudaGetLastError();
}

cudaError_t launch_grad_finish(const long long* acc, float* dense, BoxGeom g, int E, cudaStream_t stream) {
  grad_finish_kernel<<<1184, 256, 0, stream>>>(acc, dense, g, E);
  return cudaGetLastError();
}

// CTAs of a first-level reduction over n elements: one per block, at most `ctas`.
static unsigned lsqr_grid(long long n, int ctas) {
  return (unsigned)std::max(1LL, std::min<long long>((n + LSQR_BLOCK - 1) / LSQR_BLOCK, ctas));
}

// After the first-level launch over n elements (none when n = 0: the sum of nothing is +0).
static cudaError_t lsqr_finish(double* part, long long n, cudaStream_t stream, int* launches) {
  if (n == 0) return cudaMemsetAsync(part, 0, sizeof(double), stream);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  ++*launches;
  if (n <= LSQR_BLOCK) return cudaSuccess;
  lsqr_reduce_kernel<<<1, LSQR_THREADS, 0, stream>>>(part, (n + LSQR_BLOCK - 1) / LSQR_BLOCK);
  ++*launches;
  return cudaGetLastError();
}

cudaError_t launch_lsqr_sumsq(const double* p, long long n, double* part, int ctas, cudaStream_t stream, int* launches) {
  if (n > 0) lsqr_sumsq_kernel<<<lsqr_grid(n, ctas), LSQR_THREADS, 0, stream>>>(p, n, part);
  return lsqr_finish(part, n, stream, launches);
}

cudaError_t launch_lsqr_to_f32(const double* v, float* stage, long long n, cudaStream_t stream) {
  lsqr_to_f32_kernel<<<1184, 256, 0, stream>>>(v, stage, n);
  return cudaGetLastError();
}

cudaError_t launch_lsqr_u(const LsqrArgs& a, double alpha, cudaStream_t stream, int* launches) {
  const long long n = a.m + a.mD;
  if (n > 0) lsqr_u_kernel<<<lsqr_grid(n, a.ctas), LSQR_THREADS, 0, stream>>>(a, alpha);
  return lsqr_finish(a.part, n, stream, launches);
}

cudaError_t launch_lsqr_scale_u(const LsqrArgs& a, double inv_beta, cudaStream_t stream) {
  lsqr_scale_u_kernel<<<1184, LSQR_THREADS, 0, stream>>>(a, inv_beta);
  return cudaGetLastError();
}

cudaError_t launch_lsqr_v(const LsqrArgs& a, double beta, cudaStream_t stream, int* launches) {
  const long long n = (long long)a.nx * a.ny * a.nz;
  lsqr_v_kernel<<<lsqr_grid(n, a.ctas), LSQR_THREADS, 0, stream>>>(a, beta);
  return lsqr_finish(a.part, n, stream, launches);
}

cudaError_t launch_lsqr_scale(double* p, long long n, double s, cudaStream_t stream) {
  lsqr_scale_kernel<<<1184, 256, 0, stream>>>(p, n, s);
  return cudaGetLastError();
}

cudaError_t launch_lsqr_xw(const LsqrArgs& a, double t1, double t2, double inv_rho, cudaStream_t stream, int* launches) {
  const long long n = (long long)a.nx * a.ny * a.nz;
  lsqr_xw_kernel<<<lsqr_grid(n, a.ctas), LSQR_THREADS, 0, stream>>>(a, t1, t2, inv_rho);
  return lsqr_finish(a.part, n, stream, launches);
}

template <int NB>
static size_t locate_smem(int nsta) { return (size_t)nsta * 32 * NB * sizeof(double); }

template <int NB>
static bool locate_fits(int nsta, int optin) {
  cudaFuncAttributes fa{};  // the static node tables take their share besides the staged times
  return cudaFuncGetAttributes(&fa, locate_kernel<NB>) == cudaSuccess &&
         locate_smem<NB>(nsta) + fa.sharedSizeBytes <= (size_t)optin;
}

int locate_nodes_per_thread(int nsta, int device) {
  int optin = 0;
  if (cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device) != cudaSuccess) return 0;
  return locate_fits<4>(nsta, optin) ? 4 : locate_fits<2>(nsta, optin) ? 2 : locate_fits<1>(nsta, optin) ? 1 : 0;
}

template <int NB>
static cudaError_t launch_locate_nb(const LocateArgs& a, cudaStream_t stream) {
  const size_t smem = locate_smem<NB>(a.nsta);
  cudaError_t e = cudaFuncSetAttribute(locate_kernel<NB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  const long long D = (long long)a.g.nx * a.g.ny * a.g.nz;
  locate_kernel<NB><<<(unsigned)((D + 32 * NB - 1) / (32 * NB)), LOC_THREADS, smem, stream>>>(a);
  return cudaGetLastError();
}

cudaError_t launch_locate(const LocateArgs& a, int nodes_per_thread, cudaStream_t stream) {
  switch (nodes_per_thread) {
    case 4: return launch_locate_nb<4>(a, stream);
    case 2: return launch_locate_nb<2>(a, stream);
    case 1: return launch_locate_nb<1>(a, stream);
    default: return cudaErrorInvalidValue;
  }
}

cudaError_t launch_locate_finish(const LocateArgs& a, int nev, cudaStream_t stream) {
  locate_finish_kernel<<<(nev + 127) / 128, 128, 0, stream>>>(a, nev);
  return cudaGetLastError();
}

cudaError_t launch_misfit_box(const LocateArgs& a, float* dense, cudaStream_t stream) {
  misfit_box_kernel<<<1184, 256, 0, stream>>>(a, dense);
  return cudaGetLastError();
}

cudaError_t launch_fill(float* p, long long n, float value, cudaStream_t stream) {
  // boxes are multiples of 4 floats and 16-byte aligned by construction
  fill_kernel<<<1184, 256, 0, stream>>>(reinterpret_cast<float4*>(p), n / 4, value);
  return cudaGetLastError();
}
cudaError_t launch_pad_box(const float* dense, float* padded, BoxGeom g, cudaStream_t stream) {
  pad_kernel<<<1184, 256, 0, stream>>>(dense, padded, g);
  return cudaGetLastError();
}
cudaError_t launch_unpad_box(const float* padded, float* dense, BoxGeom g, cudaStream_t stream) {
  unpad_kernel<<<1184, 256, 0, stream>>>(padded, dense, g);
  return cudaGetLastError();
}
__global__ void init_state_kernel(SolveState* S, int max_rounds) {
  SolveState z = {};
  z.max_rounds = max_rounds;
  z.kmin_bits = 0x7f800000u;
  z.kmin_pub = 0x7f800000u;
  *S = z;
}
cudaError_t launch_reset_state_only(SolveState* st, int max_rounds, cudaStream_t stream) {
  init_state_kernel<<<1, 1, 0, stream>>>(st, max_rounds);
  return cudaGetLastError();
}
cudaError_t launch_fill_tmax(const RelaxArgs& a, cudaStream_t stream) {
  const size_t total = (size_t)a.nsrc * a.g.ntx * a.g.nty * a.g.ntz;
  fill_u32_kernel<<<(unsigned)std::min<size_t>(1184, (total + 255) / 256), 256, 0, stream>>>(a.tmax, (long long)total, 0x7f800000u);
  return cudaGetLastError();
}
cudaError_t launch_reset_part(const RelaxArgs& a, int max_rounds, cudaStream_t stream) {
  init_state_kernel<<<1, 1, 0, stream>>>(a.st, max_rounds);
  const size_t total = (size_t)a.nsrc * a.g.ntx * a.g.nty * a.g.ntz;
  fill_u32_kernel<<<(unsigned)std::min<size_t>(1184, (total + 255) / 256), 256, 0, stream>>>(a.key, (long long)total, 0x7f800000u);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  if (a.tmax != nullptr) {
    e = launch_fill_tmax(a, stream);
    if (e != cudaSuccess) return e;
  }
  return cudaSuccess;
}
cudaError_t launch_init_sources(const RelaxArgs& a, cudaStream_t stream) {
  init_sources_kernel<<<a.nsrc, 64, 0, stream>>>(a);
  return cudaGetLastError();
}
cudaError_t launch_reset(const RelaxArgs& a, int max_rounds, cudaStream_t stream) {
  init_state_kernel<<<1, 1, 0, stream>>>(a.st, max_rounds);
  cudaError_t e = launch_fill(a.tt, (long long)a.nsrc * a.g.vol, std::numeric_limits<float>::infinity(), stream);
  if (e != cudaSuccess) return e;
  const size_t total = (size_t)a.nsrc * a.g.ntx * a.g.nty * a.g.ntz;
  // keys: exact-length scalar fill (group slices are neither 16-byte aligned nor padded)
  fill_u32_kernel<<<(unsigned)std::min<size_t>(1184, (total + 255) / 256), 256, 0, stream>>>(a.key, (long long)total, 0x7f800000u);
  e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  if (a.tmax != nullptr) {
    e = launch_fill_tmax(a, stream);
    if (e != cudaSuccess) return e;
  }
  init_sources_kernel<<<a.nsrc, 64, 0, stream>>>(a);
  return cudaGetLastError();
}

}  // namespace sweeptt
