// pullstar.h -- host-side edge-set analysis shared by the solver and the C ABI.
//
// The reference relaxes BOTH directions of an edge from the sweep centre
// (serial_new/sweep-tt-multistart.c:222-249) but (quirk 1) never uses the last star
// entry as a centre offset (:160 passes starsize-1) and (quirk 2) skips every visit whose
// centre is the start point (:219-221).  For owner-computes GPU kernels we need the
// equivalent PULL form: for node n, which neighbours m = n+o may lower tt[n], with which
// half-distance, and which of those pulls are invalid when m is the start point.
#pragma once
#include <cmath>
#include <cstdint>
#include <vector>

#include "../../include/sweeptt.h"

namespace sweeptt {

struct PullOffset {
  int i, j, k;   // m = n + (i,j,k)
  float hd;      // 0.5f * d   (hd*(v_n+v_m) == d*(v_n+v_m)/2.0 inside the domain of DESIGN §1)
  int guarded;   // 1: only supplied by "centre m relaxes neighbour n" => invalid when m == start
};

// One (i,j) column of plain (unguarded) pulls for the tiled kernel: the k offsets present
// are a bit mask over k in [-KHALO, +KHALO]; hd values follow in ascending-k order.
struct PullColumn {
  int i, j;
  uint32_t kmask;   // bit (k + KHALO)
  int hd_begin;     // index of the first hd of this column in PullStar::col_hd
};

constexpr int KHALO = 8;      // z halo kept in shared memory / padding (16-byte aligned)
constexpr int RXY_MAX = 7;    // largest |i|,|j| the tiled kernel's shared-memory halo holds

struct PullStar {
  std::vector<PullOffset> all;       // every pull (plain first, then guarded/extra)
  std::vector<PullColumn> columns;   // plain pulls grouped by (i,j), sorted by (i,j)
  std::vector<float> col_hd;         // hd of the column-grouped pulls
  std::vector<PullOffset> extra;     // pulls handled one at a time (guarded or duplicates)
  int rx = 0, ry = 0, rz = 0;        // max |i|, |j|, |k| over all pulls
  float dmax = 0.f;                  // largest d of the star's edges (0 if none)
  float dpos = HUGE_VALF;            // smallest positive d of the star's edges (+INF if none)
  int bad_d = -1;                    // first used entry whose d is negative, NaN or infinite (-1: none)
  bool fits_tiled() const { return rx <= RXY_MAX && ry <= RXY_MAX && rz <= KHALO; }
};

// star_used <= 0 means starsize-1 (what the reference passes).
PullStar build_pull_star(const FS* fs, int starsize, int star_used);

// In-bounds pull evaluations of one round over the sub-box [x0,x1)x[y0,y1)x[z0,z1) of an
// nx*ny*nz grid (neighbour anywhere in the grid).
long long count_pulls(const PullStar& ps, int nx, int ny, int nz, int x0, int x1, int y0, int y1,
                      int z0, int z1);

// Share the star's columns out between the tiled kernel's warps.  `kmasks[c]` = k pattern of column c (its cost
// is popcount + 1.5), `gbeg` = first column of every column group (+ end).  Six tables of cut points
// (psplit[(table * max_groups + g) * (max_warps + 1) + part] = first column of the part's contiguous piece of
// group g): table % 3 == 0 spreads a group over all nw warps (tile with one live unit), 1 and 2 over the warps of
// unit 0 (warps [0, nw/2)) and unit 1 (warps [nw/2, nw)); tables 0-2 use bias[0], tables 3-5 bias[1] =
// {owner, feeder, finisher} head starts in cost units (owner = part 0 of a table, feeder = warp nw/2-1,
// finisher = warp nw-1).  loads (optional): resulting cost per (table, part), bias included.
// default head starts {owner, feeder, finisher}: [0] round-based kernels, [1] single-launch kernels, whose finisher
// also issues two device-wide fences per tile (measured on config 2: 6/2/50 -> 12.9 ms, 10/2/60 -> 12.7 ms)
constexpr double kDefaultBias[2][3] = {{8.0, 2.0, 14.0}, {10.0, 2.0, 60.0}};

// `unit_range` (optional): for unit 0 and unit 1 of the tile, per column group the sub-range [first, end) of columns
// that can reach a node inside the grid at all (tiles at the x boundary of the box: the other columns pull from
// outside the grid for every lane of the unit and are left out); tables 0, 1, 3, 4 follow unit 0, tables 2, 5 unit 1.
struct GroupRange { std::vector<int> first, end; };
void split_columns(const std::vector<uint32_t>& kmasks, const std::vector<int>& gbeg, int nw, int max_groups,
                   int max_warps, const double bias[2][3], std::vector<unsigned short>* psplit,
                   std::vector<double>* loads, double column_overhead = 1.5, const GroupRange* unit_range = nullptr);

}  // namespace sweeptt
