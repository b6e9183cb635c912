// Test-only host build of the filtered call's predicates (icikt_edges.cuh is __host__ __device__), so the
// prefilter the selection kernel runs can be checked on the CPU.
#include "../icikendalltau_b200/csrc/icikt_edges.cuh"

extern "C" void prefilter_host(long long m, const double* raw, const double* t, const double* m_sofar,
                               unsigned char* keep) {
  for (long long k = 0; k < m; ++k) keep[k] = icikt::edge_prefilter(raw[k], t[k], m_sofar[k]) ? 1 : 0;
}

extern "C" void keep_final_host(long long m, const double* raw, const double* t, int scale_max, const double* M,
                                unsigned char* keep) {
  for (long long k = 0; k < m; ++k) keep[k] = icikt::edge_keep_final(raw[k], t[k], scale_max != 0, M[k]) ? 1 : 0;
}

extern "C" int keep_window_host(int status, double raw, double pvalue, double t, double a, int scale_max,
                                double m_sofar) {
  return icikt::edge_keep_window(status, raw, pvalue, t, a, scale_max != 0, m_sofar) ? 1 : 0;
}

extern "C" long long edge_row_size() { return (long long)sizeof(icikt::EdgeRow); }
