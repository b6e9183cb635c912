// Test-only host build of p.adjust's per-rank values, scans and BY sum (icikt_padj.cuh is __host__ __device__), so
// the arithmetic the device kernels run can be checked on the CPU against the NumPy restatement of R.
#include "../icikendalltau_b200/csrc/icikt_padj.cuh"

// out[i] = the adjusted value at ascending position i of sorted[0, K), m tests: the per-rank value, R's sequential
// cummax from rank 1 up or cummin from rank K down, then pmin(1, .)
extern "C" void padj_sorted_host(int method, long long m, long long K, const double* sorted, double q, double* out) {
  for (long long i = 0; i < K; ++i) out[i] = icikt::padj_rank_value(method, m, i + 1, sorted[i], q);
  if (icikt::padj_scan_up(method)) {
    for (long long i = 1; i < K; ++i) out[i] = out[i] > out[i - 1] ? out[i] : out[i - 1];
  } else {
    for (long long i = K - 2; i >= 0; --i) out[i] = out[i] < out[i + 1] ? out[i] : out[i + 1];
  }
  for (long long i = 0; i < K; ++i) out[i] = icikt::padj_pmin1(out[i]);
}

extern "C" double padj_by_q_host(long long m) { return icikt::padj_by_q(m); }

extern "C" unsigned long long padj_key_host(double p) { return icikt::padj_key(p); }
