// icikt_common.cuh -- shared types and the fp64 epilogue of the ICI-Kendall-tau path.
//
// The epilogue restates src/kendallc.cpp:190-244 (guards) and :280-335 (tau, tau_max,
// variance, z, p-value) of the reference in terms of per-column tie statistics and the
// three per-pair integers (dis, ntie, b); SURVEY.md 7.1 derives why one set of global
// counts serves both perspectives.  It is __host__ __device__ so the same code is unit
// tested on the CPU (tests/test_epilogue_cpu.py) and run by the K3 kernel.
#pragma once
#include <cmath>
#include <cstdint>

#if defined(__CUDACC__)
#define ICIKT_HD __host__ __device__ __forceinline__
#else
#define ICIKT_HD inline
#endif

namespace icikt {

// Per-column by-products of the preprocessing kernels (K1).  Groups are the tie groups of
// the column after missing-value substitution, in ascending order; if the column has
// missing values group 0 is the "NA group" (missing rows rank below every value,
// src/kendallc.cpp:214-219), which may also hold `g0extra` non-missing rows when
// min - 0.1 == min in fp64 (SURVEY.md 8a row 3).
struct ColStats {
  int32_t n_na;       // a: missing rows
  int32_t first_run;  // size of the first group if > 1, else 0
  int32_t n_tied;     // rows in tie groups of size > 1 other than the first group
  int32_t n_groups;   // K: number of groups (distinct values, NA group included)
  int32_t levels;     // L = max(1, ceil(log2 K)): bits of a dense rank
  int32_t g0extra;    // non-missing rows merged into the NA group
  int32_t flags;      // bit 0: the missing rows tie with the minimum; bits 8..: number of large tie groups
  int32_t n_tgroups;  // number of tie groups of size > 1 other than the first group
  int64_t s2o;        // sum t(t-1)        over groups other than the NA group
  int64_t s3o;        // sum t(t-1)(t-2)
  int64_t s5o;        // sum t(t-1)(2t+5)
  uint64_t cconst;    // pass-A correction constant (see icikt_pairs.cu)
};

// Tie groups (other than the first) of at least this many rows are "large": the pair kernel
// writes them into the sequence already sorted by the other column (rank histogram, like the
// first group); the rows of the smaller groups are compared directly inside their group.  In the
// tied-row list the rows of large groups carry kLargeFlag in their group index.
constexpr int kLargeTie = 128;
// ... unless all such groups of a column are cheap enough to compare directly as well: sum of
// size^2 over them at most kDirectBudget * n (then the column has no "large" groups at all and
// can stay in the light launch tier)
constexpr int kDirectBudget = 24;
constexpr int kLargeStride = 1024;  // u16 per column in the large-group table: (start, size) x 512
constexpr unsigned kLargeFlag = 0x8000u;

// A unit of pair work: column `col` is staged in shared memory and correlated with
// `count` other columns; results go to slots [slot0, slot0+count).
struct PairUnit {
  int64_t slot0;
  int32_t col;    // staged column
  int32_t j0;     // other column of the first pair; the k-th pair uses j0 + k (j_explicit == 0)
  int32_t count;
  int32_t j_explicit;  // 1: other columns are pj_list[slot0 + k]
};

struct PairOut {
  double tau, pvalue, taumax, completeness;
  int64_t xtie, ytie, tot, n_entry, ntie;
  int32_t status;
};

// ---- R nmath pnorm_both (Cody 1969), as reached from src/kendallc.cpp:324-330 ----------
// i_tail 0 = lower only, 1 = upper only.
ICIKT_HD void pnorm_both(double x, double* cum, double* ccum, int i_tail) {
  const double a[5] = {2.2352520354606839287, 161.02823106855587881, 1067.6894854603709582,
                       18154.981253343561249, 0.065682337918207449113};
  const double b[4] = {47.20258190468824187, 976.09855173777669322, 10260.932208618978205,
                       45507.789335026729956};
  const double c[9] = {0.39894151208813466764, 8.8831497943883759412, 93.506656132177855979,
                       597.27027639480026226,  2494.5375852903726711, 6848.1904505362823326,
                       11602.651437647350124,  9842.7148383839780218, 1.0765576773720192317e-8};
  const double d[8] = {22.266688044328115691, 235.38790178262499861, 1519.377599407554805,
                       6485.558298266760755,  18615.571640885098091, 34900.952721145977266,
                       38912.003286093271411, 19685.429676859990727};
  const double p[6] = {0.21589853405795699,   0.1274011611602473639,   0.022235277870649807,
                       0.001421619193227893466, 2.9112874951168792e-5, 0.02307344176494017303};
  const double q[5] = {1.28426009614491121,   0.468238212480865118, 0.0659881378689285515,
                       0.00378239633202758244, 7.29751555083966205e-5};
  const bool lower = i_tail != 1, upper = i_tail != 0;
  double xden, xnum, temp, del, xsq;
  *cum = 0.0;
  *ccum = 0.0;
  if (x != x) { *cum = *ccum = x; return; }
  const double eps = 2.220446049250313e-16 * 0.5;
  const double y = fabs(x);
  if (y <= 0.67448975) {
    if (y > eps) {
      xsq = x * x;
      xnum = a[4] * xsq;
      xden = xsq;
      for (int i = 0; i < 3; ++i) { xnum = (xnum + a[i]) * xsq; xden = (xden + b[i]) * xsq; }
    } else {
      xnum = xden = 0.0;
    }
    temp = x * (xnum + a[3]) / (xden + b[3]);
    if (lower) *cum = 0.5 + temp;
    if (upper) *ccum = 0.5 - temp;
  } else if (y <= 5.656854249492380195206754896838) {
    xnum = c[8] * y;
    xden = y;
    for (int i = 0; i < 7; ++i) { xnum = (xnum + c[i]) * y; xden = (xden + d[i]) * y; }
    temp = (xnum + c[7]) / (xden + d[7]);
    xsq = trunc(y * 16) / 16;
    del = (y - xsq) * (y + xsq);
    *cum = exp(-xsq * xsq * 0.5) * exp(-del * 0.5) * temp;
    *ccum = 1.0 - *cum;
    if (x > 0.) { temp = *cum; if (lower) *cum = *ccum; *ccum = temp; }
  } else if ((lower && -37.5193 < x && x < 8.2924) || (upper && -8.2924 < x && x < 37.5193)) {
    xsq = 1.0 / (x * x);
    xnum = p[5] * xsq;
    xden = xsq;
    for (int i = 0; i < 4; ++i) { xnum = (xnum + p[i]) * xsq; xden = (xden + q[i]) * xsq; }
    temp = xsq * (xnum + p[4]) / (xden + q[4]);
    temp = (0.398942280401432677939946059934 - temp) / y;
    xsq = trunc(x * 16) / 16;
    del = (x - xsq) * (x + xsq);
    *cum = exp(-xsq * xsq * 0.5) * exp(-del * 0.5) * temp;
    *ccum = 1.0 - *cum;
    if (x > 0.) { temp = *cum; if (lower) *cum = *ccum; *ccum = temp; }
  } else {
    if (x > 0) { *cum = 1.; *ccum = 0.; } else { *cum = 0.; *ccum = 1.; }
  }
}

ICIKT_HD double pnorm_std(double x, bool lower_tail) {
  if (x != x) return x;
  if (fabs(x) > 1.7976931348623157e308) return ((x < 0) == lower_tail) ? 0.0 : 1.0;  // +-Inf
  double p, cp;
  pnorm_both(x, &p, &cp, lower_tail ? 0 : 1);
  return lower_tail ? p : cp;
}

ICIKT_HD double qnan() { return nan(""); }

// (double)(1.0L - (long double)m / (long double)n) bit for bit as x87 extended precision evaluates
// it -- the reference's completeness (src/kendallc.cpp:205-212: `long double completeness =
// 1 - (missingness / either_na_length)`, stored into a double) on x86-64: the quotient rounded to a
// 64-bit significand, the difference rounded to 64 bits again, then to double.  For pairs with few
// complete rows the cancellation makes this differ from the correctly rounded (n - m) / n by a few
// ulps, so it is reproduced with integer arithmetic instead.  0 <= m <= n < 2^31.
ICIKT_HD double one_minus_ratio_x87(uint64_t m, uint64_t n) {
  if (m == 0) return 1.0;
  if (m >= n) return 0.0;
  int e = 0;
  uint64_t mm = m;
  while (mm < n) {  // m/n in [2^-e, 2^-(e-1)), n <= mm < 2n
    mm <<= 1;
    ++e;
  }
  // Q = round-to-nearest-even(mm * 2^63 / n), 2^63 <= Q < 2^64: long division in base 2^32
  const uint64_t lo = (mm & 1ull) << 63;
  uint64_t r = mm >> 1;  // < n
  const uint64_t d1 = (r << 32) | (lo >> 32), q1 = d1 / n;
  r = d1 - q1 * n;
  const uint64_t d2 = (r << 32), q2 = d2 / n;  // the low 32 bits of the dividend are zero
  r = d2 - q2 * n;
  uint64_t Q = (q1 << 32) | q2;
  if (2 * r > n || (2 * r == n && (Q & 1ull))) ++Q;
  // 1 - Q * 2^-(63+e) = D * 2^-(63+e) with D = (2^k - 1) * 2^64 + L, k = e - 1, L = 2^64 - Q:
  // D has 64 + k bits, the low k are rounded away (nearest even); the result is kept * 2^-64
  const uint64_t L = 0ull - Q;
  const int k = e - 1;
  uint64_t kept = L;
  if (k > 0) {
    const uint64_t dropped = L & ((1ull << k) - 1ull), half = 1ull << (k - 1);
    kept = (~0ull << (64 - k)) | (L >> k);
    if (dropped > half || (dropped == half && (kept & 1ull))) {
      if (++kept == 0ull) return 1.0;
    }
  }
#ifdef __CUDA_ARCH__
  return __ull2double_rn(kept) * 5.421010862427522170037e-20;  // 2^-64, exact scaling
#else
  return (double)kept * 5.421010862427522170037e-20;  // u64 -> double rounds to nearest even
#endif
}

// tau, tau_max and the variance-based p-value from the exact integer counts of one pair
// (src/kendallc.cpp:280-335).  s2/s3/s5 are the column's sums of t(t-1), t(t-1)(t-2), t(t-1)(2t+5)
// over its tie groups on the np rows that enter.  Sets status 4 and returns false if every pair
// of rows is tied in x or in y (:291-298).
ICIKT_HD bool tau_from_counts(int64_t np, int64_t xs2, int64_t xs3, int64_t xs5, int64_t ys2, int64_t ys3,
                              int64_t ys5, int64_t ntie, int64_t dis, int alternative, int continuity,
                              PairOut& o) {
  // count_rank_tie, :103-118 (sums are exact int64 here; the reference's are int32)
  const int64_t xtie = xs2 / 2, ytie = ys2 / 2;
  const double x0 = (double)(xs3 / 2), y0 = (double)(ys3 / 2);
  const double x1 = (double)xs5, y1 = (double)ys5;
  o.ntie = ntie;
  const int64_t tot = np * (np - 1) / 2;  // :280
  o.xtie = xtie;
  o.ytie = ytie;
  o.tot = tot;
  if (xtie == tot || ytie == tot) { o.status = 4; return false; }  // :291-298
  // :300-308
  const double dxt = (double)xtie, dyt = (double)ytie;
  const double den = sqrt(((double)tot - dxt) * ((double)tot - dyt));
  const double con_minus_dis = (double)(tot - xtie - ytie + ntie - 2 * dis);
  const double con_plus_dis = (double)(tot - xtie - ytie + ntie);
  double tau = con_minus_dis / den;
  const double tau_max = con_plus_dis / den;
  if (tau > 1) tau = 1; else if (tau < -1) tau = -1;
  // :310-321
  const int64_t m = np * (np - 1);
  const double var = ((double)(m * (2 * np + 5)) - x1 - y1) / 18 + (2 * dxt * dyt) / (double)m +
                     x0 * y0 / (double)(9 * m * (np - 2));
  double s_adj = tau * sqrt(((double)(m / 2) - dxt) * ((double)(m / 2) - dyt));
  if (continuity) {
    const double sg = s_adj > 0 ? 1.0 : (s_adj == 0 ? 0.0 : -1.0);
    s_adj = sg * (fabs(s_adj) - 1);
  }
  const double z = s_adj / sqrt(var);
  // :323-332
  double pv = 0.0;
  if (alternative == 1) pv = pnorm_std(z, true);
  else if (alternative == 2) pv = pnorm_std(z, false);
  else if (alternative == 0) {
    const double p0 = pnorm_std(z, true), p1 = pnorm_std(z, false);
    double mn = p0;  // Rcpp sugar min(): first NaN wins
    if (mn == mn) { if (p1 != p1) mn = p1; else if (p1 < mn) mn = p1; }
    pv = 2 * mn;
  }
  o.tau = tau;
  o.pvalue = pv;
  o.taumax = tau_max;
  return true;
}

// One pair's results from the integer counts.
//   n        : vector length (features)
//   X, Y     : per-column statistics of the two columns
//   dis      : #{(p,q): x_p < x_q and y_p > y_q}            (kendall_discordant, :70-100)
//   ntie_g   : sum over joint (x,y) tie groups g(g-1)/2 on all n rows (:261-267)
//   b        : rows missing in both columns
//   g00      : rows in the lowest tie group of both columns (== b unless a column's missing
//              rows tie with its minimum, SURVEY.md 8a row 3)
ICIKT_HD void pair_epilogue(int64_t n, const ColStats& X, const ColStats& Y, int64_t dis,
                            int64_t ntie_g, int64_t b, int64_t g00, int perspective,
                            int alternative, int continuity, PairOut& o) {
  const double NA = qnan();
  o.tau = o.pvalue = o.taumax = o.completeness = NA;
  o.xtie = o.ytie = o.tot = o.ntie = 0;
  o.status = 0;
  const int64_t bb = (perspective == 1) ? b : 0;  // local drops the joint-missing rows (:180-185)
  const int64_t np = n - bb;
  o.n_entry = np;
  const int64_t a = X.n_na, c = Y.n_na;
  if (a == n || c == n) { o.status = 1; return; }  // :190-199 (a-bb == n-bb  <=>  a == n)
  if (np < 2) { o.status = 2; return; }            // :224-231
  // group 0 after removing the joint-missing rows
  const int64_t t0x = (a > 0) ? (a - bb) + X.g0extra : 0;
  const int64_t t0y = (c > 0) ? (c - bb) + Y.g0extra : 0;
  const int64_t kx = (int64_t)X.n_groups - (a > 0 ? 1 : 0) + (t0x > 0 ? 1 : 0);
  const int64_t ky = (int64_t)Y.n_groups - (c > 0 ? 1 : 0) + (t0y > 0 ? 1 : 0);
  if (kx == 1 || ky == 1) { o.status = 3; return; }  // :234-244
  // the joint group (lowest x group, lowest y group) shrinks from g00 to g00 - bb rows
  const int64_t ntie = ntie_g - g00 * (g00 - 1) / 2 + (g00 - bb) * (g00 - bb - 1) / 2;
  if (!tau_from_counts(np, X.s2o + t0x * (t0x - 1), X.s3o + t0x * (t0x - 1) * (t0x - 2),
                       X.s5o + t0x * (t0x - 1) * (2 * t0x + 5), Y.s2o + t0y * (t0y - 1),
                       Y.s3o + t0y * (t0y - 1) * (t0y - 2), Y.s5o + t0y * (t0y - 1) * (2 * t0y + 5), ntie,
                       dis, alternative, continuity, o))
    return;
  // :205-212  completeness = 1 - card(NA_x or NA_y) / length in long double, stored as double
  const int64_t miss = a + c - b - bb;
  o.completeness = one_minus_ratio_x87((uint64_t)miss, (uint64_t)np);
}

// Counts of one pair restricted to the rows present in BOTH columns (kt_fast with
// use = "pairwise.complete.obs": kt_split drops the rows missing in either column and calls
// ici_kt on what is left, R/kendalltau.R:323-341).  Produced by the pair kernel in its
// complete-observations mode from the global counts, two rank histograms and the group-start
// tables; x/y are the kernel's streamed / staged column (tau is symmetric in them).
struct PairComplete {
  int64_t n_rows;           // rows present in both columns
  int64_t dis, ntie;        // discordant pairs / joint ties among those rows
  int64_t xs2, xs3, xs5;    // tie sums of x on those rows
  int64_t ys2, ys3, ys5;
  int32_t kx, ky;           // distinct values of x / y on those rows
  int32_t unsupported, pad;  // 1: a column's missing rows tie with its minimum (host path needed)
};

ICIKT_HD void pair_epilogue_complete(const PairComplete& c, int alternative, int continuity, PairOut& o) {
  const double NA = qnan();
  o.tau = o.pvalue = o.taumax = o.completeness = NA;
  o.xtie = o.ytie = o.tot = o.ntie = 0;
  o.status = 0;
  o.n_entry = c.n_rows;
  if (c.unsupported) { o.status = 9; return; }
  if (c.n_rows == 0) { o.status = 1; return; }  // kt_split leaves NA without calling ici_kt
  if (c.n_rows < 2) { o.status = 2; return; }   // :224-231
  if (c.kx == 1 || c.ky == 1) { o.status = 3; return; }  // :234-244
  if (!tau_from_counts(c.n_rows, c.xs2, c.xs3, c.xs5, c.ys2, c.ys3, c.ys5, c.ntie, c.dis, alternative,
                       continuity, o))
    return;
  o.completeness = 1.0;  // no missing value is left in the two vectors (:205-212)
}

}  // namespace icikt
