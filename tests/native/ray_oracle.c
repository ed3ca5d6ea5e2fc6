/*
 * ray_oracle.c -- TEST INFRASTRUCTURE ONLY: CPU restatement of the ray contract of
 * sweeptt_trace_rays (include/sweeptt.h), the parity checker of the device tracer.
 * tests/test_rays.py builds it as a shared library in a temporary directory and loads it with ctypes.
 *
 * It shares nothing with the product's pull star (csrc/pullstar.cpp) or the GPU code: the candidate
 * predecessors are enumerated straight from the two edge rules of the reference sweep
 * (serial_new/sweep-tt-multistart.c:222-249, offsets [0, lused)), with the reference's own edge delay (:216).
 * Build flags: -O3 -ffp-contract=off (no FMA), like oracle/Makefile.
 */
#include <math.h>
#include <stdint.h>
#include <string.h>

/* serial_new/...c:122,127: d = delta * (float)sqrt(int) */
static float star_distance(int a, int b, int c, float delta) {
  return delta * (float)sqrt((double)(a * a + b * b + c * c));
}

/* serial_new/...c:216: float*float product, then "/ 2.0" in double, rounded back to float */
static float edge_delay(float d, float va, float vb) {
  float prod = d * (va + vb);
  return (float)((double)prod / 2.0);
}

/* float -> uint32 with the same order (-0 before +0): the tie rule's "smallest tt[m]" */
static uint32_t ordered_bits(float f) {
  uint32_t u;
  memcpy(&u, &f, 4);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

/*
 * Ray from receiver (ri,rj,rk) back to the start (si,sj,sk) through the field tt.  Candidates of node n:
 * m = n + o_l (the centre n relaxes itself from m) and m = n - o_l (the centre m relaxes n), the latter
 * skipped when m is the start because the reference skips visits whose centre is the start (:219-221);
 * in-bounds m only; cand = edge_delay + tt[m].  pred(n) = the exact match (cand == tt[n]) with the smallest
 * tt[m], then the smallest index of m.  Writes up to max_nodes nodes (x,y,z), the length and tt[receiver];
 * returns the SWEEPTT_RAY_* status (0 OK, 1 UNREACHED, 2 NOT_FIXED_POINT, 3 NO_PREDECESSOR, 4 STALLED,
 * 5 TRUNCATED).
 */
int ray_oracle_trace(const float *v, const float *tt, int nx, int ny, int nz, const int32_t *ijk, int lused,
                     float delta, int si, int sj, int sk, int ri, int rj, int rk, int max_nodes, int32_t *nodes,
                     int32_t *length_out, float *tt_out) {
  const long long sy = nz, sx = (long long)ny * nz;
  const long long src = si * sx + sj * sy + sk;
  int x = ri, y = rj, z = rk, len = 1, status;
  long long n = x * sx + y * sy + z;
  float tn = tt[n];
  *tt_out = tn;
  nodes[0] = x; nodes[1] = y; nodes[2] = z;
  if (tn == INFINITY) {
    status = 1;
  } else {
    for (;;) {
      if (n == src) { status = 0; break; }
      int below = 0, found = 0, bx = 0, by = 0, bz = 0;
      uint32_t bkey = 0;
      long long bm = 0;
      for (int l = 0; l < lused; ++l) {
        const int a = ijk[3 * l], b = ijk[3 * l + 1], c = ijk[3 * l + 2];
        if (a == 0 && b == 0 && c == 0) continue; /* self edge: no predecessor */
        const float d = star_distance(a, b, c, delta);
        for (int sgn = 1; sgn >= -1; sgn -= 2) {
          const int xo = x + sgn * a, yo = y + sgn * b, zo = z + sgn * c;
          if ((unsigned)xo >= (unsigned)nx || (unsigned)yo >= (unsigned)ny || (unsigned)zo >= (unsigned)nz)
            continue;
          const long long m = xo * sx + yo * sy + zo;
          if (sgn < 0 && m == src) continue;
          const float cand = edge_delay(d, v[n], v[m]) + tt[m];
          if (cand < tn) below = 1;
          if (cand == tn) {
            const uint32_t key = ordered_bits(tt[m]);
            if (!found || key < bkey || (key == bkey && m < bm)) {
              found = 1; bkey = key; bm = m; bx = xo; by = yo; bz = zo;
            }
          }
        }
      }
      if (below) { status = 2; break; }
      if (!found) { status = 3; break; }
      if (!(tt[bm] < tn)) { status = 4; break; }
      if (len == max_nodes) { status = 5; break; }
      x = bx; y = by; z = bz; n = bm; tn = tt[bm];
      nodes[3 * len] = x; nodes[3 * len + 1] = y; nodes[3 * len + 2] = z;
      ++len;
    }
  }
  *length_out = len;
  return status;
}

/* ray_oracle_trace for nrec receivers (rec: nrec*3); ray r's nodes at nodes[r*max_nodes*3]. */
void ray_oracle_trace_many(const float *v, const float *tt, int nx, int ny, int nz, const int32_t *ijk, int lused,
                           float delta, int si, int sj, int sk, const int32_t *rec, int nrec, int max_nodes,
                           int32_t *nodes, int32_t *length, int32_t *status, float *tt_out) {
  for (int r = 0; r < nrec; ++r)
    status[r] = ray_oracle_trace(v, tt, nx, ny, nz, ijk, lused, delta, si, sj, sk, rec[3 * r], rec[3 * r + 1],
                                 rec[3 * r + 2], max_nodes, nodes + (size_t)r * max_nodes * 3, length + r, tt_out + r);
}
