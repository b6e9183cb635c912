// icikt_padj.cuh -- R's p.adjust (stats::p.adjust) for the methods whose adjusted values a prefix of the ascending
// order determines: bonferroni, holm, hochberg, BH and BY.  __host__ __device__ so that the device kernels
// (icikt_padj.cu) and g++ (tests/padj_host.cpp) run the same arithmetic.
//
// With m the number of non-NaN p-values and p_(1) <= ... <= p_(m), R computes, in IEEE doubles and in this order:
//   bonferroni  m * p                                elementwise
//   holm        (m + 1 - i) * p_(i)                  running max from rank 1 up
//   hochberg    (m + 1 - i) * p_(i)                  running min from rank m down
//   BH          (m / i) * p_(i)                      running min from rank m down
//   BY          ((q * m) / i) * p_(i), q = sum(1/k)  running min from rank m down
// then pmin(1, .); m <= 1 returns p unchanged.  The file is compiled without contraction (--fmad=false), so every
// product and quotient here is one rounding, as in R.
//
// Ties.  Let ranks a..b hold equal p-values.  The value v(i) before the scan is g(i) * p with g non-increasing in i
// (fl(m / i), m + 1 - i and fl(fl(q m) / i) all are, rounding being monotone), so v is non-increasing over a..b.
//   * running min from the top: for i in [a, b], min(v(i..b), s(b+1)) = min(v(b), s(b+1)) = s(b);
//   * running max from the bottom: for i in [a, b], max(r(a-1), v(a..i)) = max(r(a-1), v(a)) = r(a).
// So equal p-values get equal adjusted values whatever order the sort leaves them in, the sort need not be stable,
// and a p-value finds its value at any sorted position that holds it (the lookup takes the last).
//
// Prefix.  Every multiplier is >= 1 after rounding, so padj >= p (for p <= 1, before and after pmin with 1 when
// padj <= alpha < 1).  With alpha < 1 the p-values <= alpha are a prefix of the ascending order whose ranks are the
// global ranks; a value from beyond the prefix is > alpha and can never be the running min that makes a result
// <= alpha, and the running max only looks down.  So every adjusted value <= alpha is exact when computed from the
// p-values <= alpha and m alone, and a value computed that way is > alpha exactly when the true one is.
#pragma once
#include <cmath>
#include <cstdint>
#include <cstring>

#include "icikt_common.cuh"

namespace icikt {

// method codes of include/icikt_b200.h (ICIKT_PADJ_*)
enum : int { kPadjBonferroni = 1, kPadjHolm = 2, kPadjHochberg = 3, kPadjBH = 4, kPadjBY = 5 };

// The scan direction: running max from rank 1 up (holm; bonferroni's values are non-decreasing in the rank, so the
// running max leaves them as they are), or running min from rank m down (hochberg, BH, BY).
ICIKT_HD bool padj_scan_up(int method) { return method == kPadjBonferroni || method == kPadjHolm; }

// The value at ascending rank i (1-based) of m, before the scan and pmin; q: BY's sum(1/(1:m)).
ICIKT_HD double padj_rank_value(int method, int64_t m, int64_t i, double p, double q) {
  const double dm = (double)m;
  switch (method) {
    case kPadjBonferroni: return dm * p;
    case kPadjHolm:
    case kPadjHochberg: return (double)(m + 1 - i) * p;
    case kPadjBH: return (dm / (double)i) * p;
    default: return ((q * dm) / (double)i) * p;
  }
}

ICIKT_HD double padj_pmin1(double v) { return v < 1.0 ? v : 1.0; }  // pmin(1, v) for a non-NaN v

// The sort key of a p-value: its bit pattern, so that the unsigned order is the numeric order of non-negative
// doubles; -0.0 becomes +0.0 (it would sort last otherwise).
ICIKT_HD unsigned long long padj_key(double p) {
  if (p == 0.0) p = 0.0;
#ifdef __CUDA_ARCH__
  return (unsigned long long)__double_as_longlong(p);
#else
  unsigned long long k;
  std::memcpy(&k, &p, sizeof(k));
  return k;
#endif
}

// BY's q = sum(1/(1:m)) as R forms it: every term a double 1.0 / k, summed in ascending k in a long double (R's
// rsum accumulates in LDOUBLE; on x86-64 the 80-bit x87 format), then rounded to double.  Host only; m steps.
inline double padj_by_q(int64_t m) {
  long double s = 0.0L;
  for (int64_t k = 1; k <= m; ++k) {
    const double t = 1.0 / (double)k;
    s += t;
  }
  return (double)s;
}

}  // namespace icikt
