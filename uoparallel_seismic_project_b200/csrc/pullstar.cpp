// pullstar.cpp -- see pullstar.h.  Pure host code, no CUDA.
#include "pullstar.h"

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <map>
#include <tuple>

namespace sweeptt {

namespace {
struct Key {
  int i, j, k;
  uint32_t dbits;
  bool operator<(const Key& o) const {
    return std::tie(i, j, k, dbits) < std::tie(o.i, o.j, o.k, o.dbits);
  }
};
uint32_t bits_of(float f) {
  uint32_t u;
  std::memcpy(&u, &f, 4);
  return u;
}
}  // namespace

PullStar build_pull_star(const FS* fs, int starsize, int star_used) {
  PullStar ps;
  if (star_used <= 0 || star_used > starsize) star_used = starsize - 1;
  // (offset, distance) -> is the pull supplied unconditionally (rule 1) / only by the
  // neighbour's own visit (rule 2)?
  //   rule 1: centre n, star entry l: n may take delay + tt[n+o_l]       (:233-243), n != start
  //   rule 2: centre m, star entry l: neighbour n = m+o_l may take delay + tt[m] (:228-232,
  //           :245-248), i.e. n pulls over offset -o_l, valid only while m != start (:219-221)
  std::map<Key, int> have;  // bit0 = rule 1, bit1 = rule 2
  for (int l = 0; l < star_used; ++l) {
    const FS& e = fs[l];
    if (e.i == 0 && e.j == 0 && e.k == 0) continue;  // self edge: can never change anything
    if (!(e.d >= 0.f) || std::isinf(e.d)) {  // negative or NaN, or infinite
      if (ps.bad_d < 0) ps.bad_d = l;
    } else {
      ps.dmax = std::max(ps.dmax, e.d);
      if (e.d > 0.f) ps.dpos = std::min(ps.dpos, e.d);
    }
    have[Key{e.i, e.j, e.k, bits_of(e.d)}] |= 1;
    have[Key{-e.i, -e.j, -e.k, bits_of(e.d)}] |= 2;
  }
  std::vector<PullOffset> plain;
  for (const auto& kv : have) {
    PullOffset p;
    p.i = kv.first.i; p.j = kv.first.j; p.k = kv.first.k;
    float d;
    std::memcpy(&d, &kv.first.dbits, 4);
    p.hd = d * 0.5f;
    p.guarded = (kv.second & 1) ? 0 : 1;  // rule 1 subsumes rule 2 (tt[start] is never updated)
    ps.rx = std::max(ps.rx, std::abs(p.i));
    ps.ry = std::max(ps.ry, std::abs(p.j));
    ps.rz = std::max(ps.rz, std::abs(p.k));
    if (p.guarded) ps.extra.push_back(p); else plain.push_back(p);
  }
  // Column grouping of the plain pulls.  A second plain pull with the same (i,j,k) but a
  // different distance (only possible for hand-made stars) goes to the one-at-a-time list.
  std::map<std::pair<int, int>, std::vector<PullOffset>> cols;
  std::vector<PullOffset> grouped;
  for (const auto& p : plain) {
    auto& col = cols[{p.i, p.j}];
    bool dup = false;
    for (const auto& q : col) dup |= (q.k == p.k);
    if (dup || std::abs(p.k) > KHALO) ps.extra.push_back(p); else col.push_back(p);
  }
  for (auto& kv : cols) {
    auto& col = kv.second;
    if (col.empty()) continue;
    std::sort(col.begin(), col.end(), [](const PullOffset& a, const PullOffset& b) { return a.k < b.k; });
    PullColumn c;
    c.i = kv.first.first; c.j = kv.first.second; c.kmask = 0;
    c.hd_begin = (int)ps.col_hd.size();
    for (const auto& p : col) {
      c.kmask |= 1u << (p.k + KHALO);
      ps.col_hd.push_back(p.hd);
      grouped.push_back(p);
    }
    ps.columns.push_back(c);
  }
  ps.all = grouped;
  ps.all.insert(ps.all.end(), ps.extra.begin(), ps.extra.end());
  return ps;
}

long long count_pulls(const PullStar& ps, int nx, int ny, int nz, int x0, int x1, int y0, int y1,
                      int z0, int z1) {
  auto span = [](int lo, int hi, int o, int n) -> long long {
    // #{c in [lo,hi) : 0 <= c+o < n}
    int a = std::max(lo, -o), b = std::min(hi, n - o);
    return b > a ? (long long)(b - a) : 0;
  };
  x1 = std::min(x1, nx); y1 = std::min(y1, ny); z1 = std::min(z1, nz);
  long long total = 0;
  for (const auto& p : ps.all)
    total += span(x0, x1, p.i, nx) * span(y0, y1, p.j, ny) * span(z0, z1, p.k, nz);
  return total;
}

void split_columns(const std::vector<uint32_t>& kmasks, const std::vector<int>& gbeg, int nw, int max_groups,
                   int max_warps, const double bias[2][3], std::vector<unsigned short>* psplit,
                   std::vector<double>* loads_out, double column_overhead, const GroupRange* unit_range) {
  const int ngroups = (int)gbeg.size() - 1;
  const int feeder = nw / 2 - 1, finisher = nw - 1;  // warp indices (kernels.cu)
  auto cost = [&](int col) { return (double)__builtin_popcount(kmasks[col]) + column_overhead; };
  psplit->assign((size_t)6 * max_groups * (max_warps + 1), 0);
  if (loads_out) loads_out->assign((size_t)6 * max_warps, 0.0);
  for (int table = 0; table < 6; ++table) {  // 0-2: round-based kernels, 3-5: single-launch kernels
    const int parts = table % 3 == 0 ? nw : nw / 2;
    const int warp0 = table % 3 == 2 ? nw / 2 : 0;  // first warp of this table's unit
    const double b_own = bias[table / 3][0], b_feed = bias[table / 3][1], b_fin = bias[table / 3][2];
    std::vector<double> load(parts, 0.0);
    for (int pt = 0; pt < parts; ++pt) {
      const int w = warp0 + pt;
      if (pt == 0) load[pt] += b_own;
      if (w == feeder) load[pt] += b_feed;
      if (w == finisher) load[pt] += b_fin;
    }
    const GroupRange* ur = unit_range ? &unit_range[table % 3 == 2 ? 1 : 0] : nullptr;
    for (int g = 0; g < ngroups && g < max_groups; ++g) {
      const int gfirst = ur ? ur->first[g] : gbeg[g], gend = ur ? ur->end[g] : gbeg[g + 1];
      double gcost = 0;
      for (int col = gfirst; col < gend; ++col) gcost += cost(col);
      double total = gcost;
      for (double l : load) total += l;
      // water-filling level: parts already above it get nothing from this group
      double level = total / parts;
      for (int iter = 0; iter < parts; ++iter) {
        double sum = gcost;
        int n = 0;
        for (double l : load) if (l < level) { sum += l; ++n; }
        const double nl = n ? sum / n : level;
        if (std::fabs(nl - level) < 1e-9) break;
        level = nl;
      }
      unsigned short* row = &(*psplit)[((size_t)table * max_groups + g) * (max_warps + 1)];
      // columns per part: its deficit below the level in units of the group's mean column cost, rounded by
      // largest remainder so that the counts add up (what rounding costs a part here it gets back from
      // the next groups, because the level is recomputed from the actual loads)
      const int n = gend - gfirst;
      const double wavg = gcost / std::max(1, n);
      std::vector<int> cntp(parts, 0);
      std::vector<std::pair<double, int>> frac;
      int given = 0;
      for (int pt = 0; pt < parts; ++pt) {
        const double x = std::max(0.0, level - load[pt]) / wavg;
        cntp[pt] = (int)std::floor(x);
        given += cntp[pt];
        frac.push_back({x - std::floor(x), pt});
      }
      std::sort(frac.begin(), frac.end(), [](const std::pair<double, int>& a, const std::pair<double, int>& b) {
        return a.first > b.first || (a.first == b.first && a.second < b.second);
      });
      for (int i = 0; given < n; i = (i + 1) % parts) { cntp[frac[i].second] += 1; ++given; }
      for (int i = parts - 1; given > n; i = (i + parts - 1) % parts)
        if (cntp[frac[i].second] > 0) { cntp[frac[i].second] -= 1; --given; }
      int col = gfirst;
      for (int pt = 0; pt < parts; ++pt) {
        row[pt] = (unsigned short)col;
        for (int k = 0; k < cntp[pt]; ++k, ++col) load[pt] += cost(col);
      }
      for (int pt = parts; pt <= max_warps; ++pt) row[pt] = (unsigned short)gend;
    }
    if (loads_out)
      for (int pt = 0; pt < parts; ++pt) (*loads_out)[(size_t)table * max_warps + pt] = load[pt];
  }
}

}  // namespace sweeptt

// Test hook (tests/test_pullstar.py): the column split of a star for `nw` warps, one pattern group per distinct
// k mask, default head starts.  Writes 6 * ngroups * (nw + 1) cut points, returns the number of columns or -1.
extern "C" int sweeptt_debug_column_split(const struct FS* fs, int starsize, int nw, int* ngroups_out,
                                          unsigned short* cuts, int cuts_capacity, unsigned* kmasks_out,
                                          int kmasks_capacity) {
  using namespace sweeptt;
  PullStar ps = build_pull_star(fs, starsize, 0);
  std::stable_sort(ps.columns.begin(), ps.columns.end(),
                   [](const PullColumn& a, const PullColumn& b) { return a.kmask < b.kmask; });
  std::vector<uint32_t> kmasks;
  std::vector<int> gbeg;
  for (size_t i = 0; i < ps.columns.size(); ++i) {
    if (i == 0 || ps.columns[i].kmask != ps.columns[i - 1].kmask) gbeg.push_back((int)i);
    kmasks.push_back(ps.columns[i].kmask);
  }
  gbeg.push_back((int)ps.columns.size());
  const int ngroups = (int)gbeg.size() - 1;
  std::vector<unsigned short> psplit;
  split_columns(kmasks, gbeg, nw, ngroups, nw, kDefaultBias, &psplit, nullptr);
  if ((int)psplit.size() > cuts_capacity || (int)kmasks.size() > kmasks_capacity) return -1;
  std::copy(psplit.begin(), psplit.end(), cuts);
  std::copy(kmasks.begin(), kmasks.end(), kmasks_out);
  if (ngroups_out) *ngroups_out = ngroups;
  return (int)kmasks.size();
}
