// icikt_topk.cuh -- the ranking of the top-k all-pairs call (icikt_all_pairs_topk).  __host__ __device__ so that
// the selection kernels and the tests (tests/topk_host.cpp, tests/topk_merge_host.cpp, compiled by g++) run the
// same code.
//
// A candidate of column c is a partner d with its pair's raw.  Candidates are ranked by (key descending,
// partner ascending), a strict total order since a partner occurs once per column.  The key is a uint64 whose
// unsigned order is the order of |raw| (by = ICIKT_TOPK_ABS) or of raw (ICIKT_TOPK_SIGNED, -0.0 equal to +0.0).
#pragma once
#include <cstring>

#include "icikt_common.cuh"

namespace icikt {

ICIKT_HD unsigned long long topk_key(double raw, int by) {
  if (raw == 0.0) raw = 0.0;  // -0.0 -> +0.0
  unsigned long long b;
  memcpy(&b, &raw, sizeof(b));
  if (by == 0) return b & 0x7fffffffffffffffULL;  // non-negative doubles order as their bits
  return (b >> 63) ? ~b : (b | 0x8000000000000000ULL);
}

// does (ka, ia) come before (kb, ib)?
ICIKT_HD bool topk_before(unsigned long long ka, int32_t ia, unsigned long long kb, int32_t ib) {
  return ka > kb || (ka == kb && ia < ib);
}

// The merge-path rank of the device merge (icikt_all_pairs_topk_multi): how many entries of the sorted list
// (key, part)[0..m) come before (k0, p0).  Merging two sorted lists whose partners are disjoint, an entry lands at
// its index in its own list plus its rank in the other one; the positions are distinct since the order is strict.
ICIKT_HD int topk_rank(const unsigned long long* key, const int32_t* part, int m, unsigned long long k0, int32_t p0) {
  int lo = 0, hi = m;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (topk_before(key[mid], part[mid], k0, p0)) lo = mid + 1; else hi = mid;
  }
  return lo;
}

}  // namespace icikt
