// Test-only host build of the component calls' union-find (icikt_components.cuh is __host__ __device__): the merge of
// several devices' labels that the host runs, and a sequential run of the find and hook the tally kernel runs.
#include "../icikendalltau_b200/csrc/icikt_components.cuh"

// labels: K tables of [T][V] labels, one after the other
extern "C" void merge_host(int T, long long V, int K, const int32_t* labels, int32_t* out, long long* n_components) {
  std::vector<const int32_t*> tables;
  for (int k = 0; k < K; ++k) tables.push_back(labels + (long long)k * T * V);
  std::vector<int64_t> n((size_t)T);
  icikt::merge_component_labels(T, V, tables, out, n.data());
  for (int f = 0; f < T; ++f) n_components[f] = n[(size_t)f];
}

// the forest of V vertices after uniting the m edges (a[e], b[e]) in order; labels[v] = root, returns the hooks
extern "C" long long unite_host(long long V, long long m, const int32_t* a, const int32_t* b, int32_t* labels) {
  for (long long v = 0; v < V; ++v) labels[v] = (int32_t)v;
  long long hooks = 0;
  for (long long e = 0; e < m; ++e) hooks += icikt::uf_unite(labels, a[e], b[e]) ? 1 : 0;
  for (long long v = 0; v < V; ++v) {
    if (labels[v] > v) return -1;  // the invariant parent[v] <= v
  }
  for (long long v = 0; v < V; ++v) labels[v] = icikt::uf_root(labels, (int32_t)v);
  return hooks;
}
