// icikt_cross.cuh -- the pair order of the cross calls (icikt_cross_pairs, icikt_cross_edges, icikt_cross_topk): every
// column i of X (Cx columns) against every column j of Y (Cy columns), x-major, pair p = i * Cy + j.  The plan holds
// [X | Y] as one matrix of Cx + Cy columns, so pair (i, j) is the plan's pair (i, Cx + j), staged with X's column.
// Host code only; plain C++ so that g++ can compile it for the tests (tests/cross_host.cpp).
#pragma once
#include <algorithm>
#include <cstdint>
#include <vector>

#include "icikt_common.cuh"

namespace icikt {

// The units of pairs [lo, hi) of the cross order, appended to U with slots counted from lo.  The unit length follows
// range_units (the combn order's builder): (hi - lo) / (16 slots), clamped to [1, 16], where `slots` is the number of
// resident CTAs of the pair kernel.  A unit never crosses an x column, so every unit is one contiguous run of Y.
inline void cross_units(int64_t Cx, int64_t Cy, int64_t lo, int64_t hi, int64_t slots, std::vector<PairUnit>& U) {
  if (hi <= lo || Cy < 1) return;
  const int64_t ulen = std::max<int64_t>(1, std::min<int64_t>(16, (hi - lo) / (16 * slots)));
  for (int64_t i = lo / Cy; i < Cx && i * Cy < hi; ++i) {
    const int64_t rs = i * Cy;
    const int64_t a = std::max(rs, lo), b = std::min(rs + Cy, hi);
    for (int64_t s = a; s < b; s += ulen) {
      PairUnit u;
      u.slot0 = s - lo;
      u.col = (int32_t)i;
      u.j0 = (int32_t)(Cx + (s - rs));
      u.count = (int32_t)std::min<int64_t>(ulen, b - s);
      u.j_explicit = 0;
      U.push_back(u);
    }
  }
}

}  // namespace icikt
