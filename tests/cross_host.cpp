// Test-only host build of the cross calls' unit builder (icikt_cross.cuh), so that the units a window gets can be
// checked on the CPU.
#include "../icikendalltau_b200/csrc/icikt_cross.cuh"

// units of pairs [lo, hi) as rows (slot0, col, j0, count, j_explicit) into out[5 * cap]; returns the number of units
extern "C" long long cross_units_host(long long Cx, long long Cy, long long lo, long long hi, long long slots,
                                      long long cap, long long* out) {
  std::vector<icikt::PairUnit> U;
  icikt::cross_units(Cx, Cy, lo, hi, slots, U);
  for (size_t k = 0; k < U.size() && (long long)k < cap; ++k) {
    out[5 * k + 0] = U[k].slot0;
    out[5 * k + 1] = U[k].col;
    out[5 * k + 2] = U[k].j0;
    out[5 * k + 3] = U[k].count;
    out[5 * k + 4] = U[k].j_explicit;
  }
  return (long long)U.size();
}
