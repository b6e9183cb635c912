// icikt_edges.cuh -- the predicates of the filtered all-pairs call (icikt_all_pairs_edges).  __host__ __device__
// so that the selection kernel and the host trims run the same code, and g++ can compile it for the tests
// (tests/edges_host.cpp).
//
// A pair is an edge iff status == 0 && (isnan(t) || fabs(cor) >= t) && (isnan(a) || pvalue <= a), with
// cor = raw / M (scale_max) or raw, M = max(taumax) over all pairs.  With scale_max, M is only known after the
// last window; M_sofar <= M is known after each, and edge_prefilter keeps a superset of the final edges with it.
#pragma once
#include "icikt_common.cuh"

namespace icikt {

// Layout of one selected row (host and device).
struct EdgeRow {
  int32_t i, j;
  double raw, pvalue, taumax, completeness;
};

// Can |raw / M| >= t hold for some M >= m_sofar > 0?  If fl(raw / M) >= t >= 2^-1000, the quotient is normal, so
// |raw| >= t * M * (1 - 2^-52) >= t * m_sofar * (1 - 2^-52); the threshold computed here, fl(fl(t * m_sofar) *
// (1 - 2^-50)), is below that whenever t * m_sofar is normal, since the two roundings cost at most 2^-52 together.
// Thresholds that could be subnormal, a t outside [2^-1000, 2^1000] and a NaN t keep the pair: the result is
// always a superset, never a loss.
ICIKT_HD bool edge_prefilter(double raw, double t, double m_sofar) {
  if (!(t >= 0x1p-1000 && t <= 0x1p1000)) return true;
  const double thr = t * m_sofar * (1.0 - 0x1p-50);
  if (!(thr >= 0x1p-1000)) return true;  // also NaN (m_sofar NaN or 0 * inf)
  return fabs(raw) >= thr;
}

// The selection on the device, for a pair of a window: exact for the p-value and, without scale_max, for cor;
// with scale_max the cor condition is the prefilter against the maximum so far.
ICIKT_HD bool edge_keep_window(int32_t status, double raw, double pvalue, double t, double a, bool scale_max,
                               double m_sofar) {
  if (status != 0) return false;
  if (t == t && !(scale_max ? edge_prefilter(raw, t, m_sofar) : fabs(raw) >= t)) return false;
  return a != a || pvalue <= a;
}

// The cor condition with the final maximum M (scale_max), applied on the host after the last window.
ICIKT_HD bool edge_keep_final(double raw, double t, bool scale_max, double M) {
  const double cor = scale_max ? raw / M : raw;
  return t != t || fabs(cor) >= t;
}

}  // namespace icikt
