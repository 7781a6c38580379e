// The summation orders of the mix-down, defined once for the kernels and the CPU suite's mock device. Floating-point sums depend on
// their association, so every place that sums voices for the same mix uses these.
#pragma once
#include "bank_args.h"

namespace fdsp {

// One half (h = 0: columns [0, NT/2), h = 1: the rest) of a row of the CTA mix tile, summed with four interleaved accumulators in
// the fixed association ((a0 + a1) + (a2 + a3)); the row's sum is half 0 + half 1. The odd half starts its accumulators QN columns
// further, so that the 32 lanes of a warp (16 rows x 2 halves) hit 32 banks.
template <int NT> FDSP_HDC float cta_half_row_sum(const float* row, int h) {
  constexpr int HALF = NT / 2, QN = HALF / 4 > 0 ? HALF / 4 : 1;
  const int c0 = h * HALF + (h * QN) % HALF, c1 = h * HALF + (QN + h * QN) % HALF, c2 = h * HALF + (2 * QN + h * QN) % HALF, c3 = h * HALF + (3 * QN + h * QN) % HALF;
  float a0 = row[c0], a1 = row[c1], a2 = row[c2], a3 = row[c3];
#pragma unroll
  for (int q = 1; q < QN; q++) { a0 += row[c0 + q]; a1 += row[c1 + q]; a2 += row[c2 + q]; a3 += row[c3 + q]; }
  return (a0 + a1) + (a2 + a3);
}

// One mix element from the per-CTA partials p0[b * part_stride], b = 0 .. nparts-1: a left fold in CTA order. The loads of 8 CTAs
// are issued together (ld(p) reads one partial); the adds stay in order.
template <class Ld> FDSP_HDC float cta_order_fold(const float* p0, size_t part_stride, uint32_t nparts, Ld&& ld) {
  float s = ld(p0);
  uint32_t b = 1;
  for (; b + 8 <= nparts; b += 8) {
    float x[8];
#pragma unroll
    for (int u = 0; u < 8; u++) x[u] = ld(p0 + (size_t)(b + u) * part_stride);
#pragma unroll
    for (int u = 0; u < 8; u++) s += x[u];
  }
  for (; b < nparts; b++) s += ld(p0 + (size_t)b * part_stride);
  return s;
}

// The balanced adder tree of a reference `Net::bus` (level-wise adjacent pairing, the odd element carried up) as a binary carry
// stack st[]: carry_push adds element q (pushed in order; a complete aligned block of 2^lvl elements may be pushed as its sum, with
// q its block index, at level lvl), carry_finish folds what is left after V elements.
FDSP_HDC inline void carry_push(float* st, float y, uint32_t q, int lvl) {
  while (q & 1u) { y = st[lvl] + y; q >>= 1; lvl++; }
  st[lvl] = y;
}
FDSP_HDC inline float carry_finish(const float* st, uint32_t V) {
  int lvl = 0; uint32_t q = V;
  while (!(q & 1u)) { q >>= 1; lvl++; }
  float x = st[lvl]; q >>= 1; lvl++;
  for (; q; q >>= 1, lvl++) if (q & 1u) x = st[lvl] + x;
  return x;
}

}  // namespace fdsp
