// Test-only host build of the device merge of icikt_all_pairs_topk_multi: the fold of topk_device_merge_kernel
// (icikt_select.cu), one list at a time into an accumulator of at most k entries, with the merge-path rank of
// icikt_topk.cuh.  Every "thread" computes its new position before any entry moves, as the kernel does between
// its two barriers.
#include <vector>

#include "../icikendalltau_b200/csrc/icikt_topk.cuh"

// n_dev lists, list d at [off[d], off[d + 1]) of raw / part, each sorted best first and at most k long.
// Writes the merged list (partner, and source = device * 1024 + position) and returns its length.
extern "C" int topk_merge_host(int n_dev, const long long* off, const double* raw, const int* part, int k, int by,
                               int* out_part, int* out_src) {
  std::vector<unsigned long long> akey((size_t)k), bkey((size_t)k), nkey((size_t)k);
  std::vector<int32_t> apart((size_t)k), asrc((size_t)k), bpart((size_t)k), npart((size_t)k), nsrc((size_t)k);
  int a = 0;
  for (int d = 0; d < n_dev; ++d) {
    const int b = (int)(off[d + 1] - off[d]);
    if (b == 0) continue;
    for (int t = 0; t < b; ++t) {
      bkey[(size_t)t] = icikt::topk_key(raw[off[d] + t], by);
      bpart[(size_t)t] = part[off[d] + t];
    }
    for (int t = 0; t < a; ++t) {
      const int pa = t + icikt::topk_rank(bkey.data(), bpart.data(), b, akey[(size_t)t], apart[(size_t)t]);
      if (pa < k) {
        nkey[(size_t)pa] = akey[(size_t)t];
        npart[(size_t)pa] = apart[(size_t)t];
        nsrc[(size_t)pa] = asrc[(size_t)t];
      }
    }
    for (int t = 0; t < b; ++t) {
      const int pb = t + icikt::topk_rank(akey.data(), apart.data(), a, bkey[(size_t)t], bpart[(size_t)t]);
      if (pb < k) {
        nkey[(size_t)pb] = bkey[(size_t)t];
        npart[(size_t)pb] = bpart[(size_t)t];
        nsrc[(size_t)pb] = d * 1024 + t;
      }
    }
    a = a + b < k ? a + b : k;
    akey.swap(nkey);
    apart.swap(npart);
    asrc.swap(nsrc);
  }
  for (int t = 0; t < a; ++t) {
    out_part[t] = apart[(size_t)t];
    out_src[t] = asrc[(size_t)t];
  }
  return a;
}
