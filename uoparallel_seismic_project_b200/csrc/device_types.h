// device_types.h -- structs shared between the host solver and the sm_100a kernels.
#pragma once
#include <cstdint>

namespace sweeptt {

// ---- tile shape of the tiled kernel -------------------------------------------------
// Interior tile TX x TY x TZ nodes.  The work unit of a warp is a 4 x 8 x 8 block: lane ->
// (x within the 4-wide unit, y), each thread owns the KZ = 8 consecutive z nodes of its (x,y)
// column (register window along the fastest axis).  A tile holds UNITS = TX/4 units; the star's
// columns of every unit are shared out between the CTA's compute warps.  Small tiles keep the
// activation granularity (one key per tile) close to the star radius, which is what bounds the
// number of times a node is re-relaxed while the front crosses it.
#ifndef SWEEPTT_TX
#define SWEEPTT_TX 8
#endif
constexpr int TX = SWEEPTT_TX, TY = 8, TZ = 8, KZ = 8;
static_assert(TX == 4 || TX == 8, "a tile is one or two 4x8x8 units");
constexpr int UNITS = TX / 4;
constexpr int ZHALO = 8;                 // z halo staged on both sides (16-byte aligned)
constexpr int SZD = TZ + 2 * ZHALO + 4;  // smem/TMA row length: 28 floats; 28/4 = 7 is odd,
                                         // which makes the quarter-warp LDS.128 conflict-free
constexpr int WIN = KZ + 2 * ZHALO;      // 24-float register window per (i,j) column
#ifndef SWEEPTT_NW
#define SWEEPTT_NW 16
#endif
constexpr int MAX_WARPS = SWEEPTT_NW;    // compute warps per CTA of the 5-FS / 818-FS kernels (even; 20 = five per scheduler
                                         // needs <= 102 registers per thread)
constexpr int XREACH = (7 + TX - 1) / TX;  // tiles that a changed node (reach <= 7 nodes) can affect along x
constexpr int NMARK = (2 * XREACH + 1) * 9;

// ---- padded device float box ----------------------------------------------------------
// Logical node (x,y,z) lives at padded index ((x+AX)*py + (y+AY))*pz + (z+AZ).
// Apron: slowness = +INF (makes every edge touching it infinitely slow, which reproduces the
// reference's bounds `continue`, serial_new/sweep-tt-multistart.c:210-214, with no test in
// the inner loop), travel time = +INF.
constexpr int AX = 7, AY = 7, AZ = ZHALO;

// The kernels work in a PERMUTED coordinate system: kernel axis q is the caller's axis perm[q],
// chosen so that the register-window axis (kernel z, tiled by 32) is the caller axis that tiles
// best (241x241x51: windows run along the caller's y, 51 is tiled by 8).  The permutation lives
// only in the pad/un-pad kernels, the star offsets and the start points.
struct BoxGeom {
  int nx, ny, nz;      // logical dims in KERNEL axis order
  int perm[3];         // kernel axis q = caller axis perm[q]
  long long dstride[3];// stride (floats) of kernel axis q in the caller's dense FLOATBOX
  int px, py, pz;      // padded dims
  int ntx, nty, ntz;   // tiles per axis
  long long sx;        // py*pz
  long long vol;       // px*py*pz floats per box
};

// ---- device-resident convergence state --------------------------------------------------
struct SolveState {
  int round;                 // rounds completed so far
  int last_changed_round;    // 1-based index of the last round that changed anything
  int parity;                // which work list the next round reads
  unsigned count[2];         // entries in each work list
  unsigned cursor;           // work-stealing cursor of the running round
  unsigned ticket;           // last-block-done ticket of the compaction kernel
  unsigned long long tile_visits;
  unsigned long long pulls;  // in-bounds pull evaluations executed
  unsigned long long units_run;      // (warp, tile) units that ran the column phase
  unsigned long long units_changed;  // ... of which lowered at least one travel time
  int max_rounds;            // 0 = unlimited; the graph WHILE loop stops here
  unsigned kmin_bits;        // smallest activation key among dirty tiles (scan pass of the compaction)
  unsigned ticket2;          // last-block-done ticket of scan_min_key (one grid over several devices)
  unsigned kmin_pub;         // one grid over several devices: smallest pending key at this part's last compaction
                             // (INF: nothing pending); read by the other parts and by the host's termination test
  // ---- single-launch (persistent) scheduling: work lists come in GENERATIONS built on the device ----
  unsigned gen;              // newest published generation; its list is work list (gen & 1)
  unsigned builder;          // generation some CTA has claimed to build (== gen + 1 while a build is running)
  unsigned done;             // 1 = fixed point reached, 2 = watchdog gave up (error)
  unsigned inflight;         // tiles published on a list and not yet finished
  // generation g's list lives in slot g & 3: entry count in the HIGH word, pop cursor in the LOW word.  One
  // 64-bit word so that a pop (atomicAdd of 1) reads cursor and count of the SAME generation and the builder
  // recycles a slot with ONE store: a straggler still popping generation g-4 either sees the old, exhausted
  // pair or takes a valid entry of the new list -- never an entry that is handed out a second time.
  unsigned long long gslot[4];
};

struct ColumnDev {
  int soff;        // smem float offset of the column: i*SYD*SZD + j*SZD
  unsigned kmask;  // bit (k + ZHALO) for every k present
  int hd_begin;    // first half-distance in c_col_hd
  unsigned gmask;  // which 4-float granules of the 24-float window the column touches
};

struct ExtraDev {
  int i, j, k;
  int soff;        // smem float offset i*SYD*SZD + j*SZD + k
  float hd;
  int guarded;
  int pad0, pad1;
};

struct StarDev {   // star as the simple kernel / verifier read it (global memory)
  int i, j, k;
  float hd;
  int guarded;
};

struct RayPull {   // one candidate-predecessor offset of the ray tracer (16 bytes, one LDS.128)
  short i, j, k;         // kernel-axis offset m - n
  unsigned short rank;   // bits 0-14: position of the offset in caller-axis lexicographic order (the tie rule:
                         // for in-bounds m it orders the FLOATBOX index of m); bit 15: guarded (invalid at m == start)
  int off;               // padded-box offset of m - n
  float hd;
};
constexpr unsigned RAY_GUARD_BIT = 0x8000u;
constexpr int RAY_MAX_PULLS = 1 << 15;

constexpr int MAX_PARTS = 16;    // devices (or contexts sharing devices) that one grid can be spread over

constexpr int MAX_COLUMNS = 320;
constexpr int MAX_PATTERNS = SWEEPTT_NW > 20 ? 20 : SWEEPTT_NW > 16 ? 24 : 31;  // (the column tables must fit 64 KB of constant memory)
constexpr int MAX_COL_HD = 4096;
constexpr int MAX_EXTRA = 128;
constexpr int NXCLASS = 3;       // column tables per tile position along x: interior, first tile, last tile (kernels.cu c_pdesc)

}  // namespace sweeptt
