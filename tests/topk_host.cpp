// Test-only host build of the top-k call's ranking (icikt_topk.cuh is __host__ __device__), so the order the
// selection kernels use can be checked on the CPU.
#include <algorithm>
#include <numeric>
#include <vector>

#include "../icikendalltau_b200/csrc/icikt_topk.cuh"

extern "C" void topk_keys_host(long long m, const double* raw, int by, unsigned long long* key) {
  for (long long q = 0; q < m; ++q) key[q] = icikt::topk_key(raw[q], by);
}

// the permutation that sorts (raw, partner) by (key descending, partner ascending)
extern "C" void topk_sort_host(long long m, const double* raw, const int* partner, int by, long long* order) {
  std::vector<unsigned long long> key((size_t)m);
  topk_keys_host(m, raw, by, key.data());
  std::iota(order, order + m, 0LL);
  std::sort(order, order + m, [&](long long a, long long b) {
    return icikt::topk_before(key[(size_t)a], partner[a], key[(size_t)b], partner[b]);
  });
}
