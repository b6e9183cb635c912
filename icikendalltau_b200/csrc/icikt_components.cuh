// icikt_components.cuh -- the union-find forests of the component calls (icikt_all_pairs_components,
// icikt_cross_components).  The find and the hook are __host__ __device__: the tally kernel runs them concurrently
// on the device, the host merge of several devices' labels runs them sequentially, and g++ compiles them for the
// tests (tests/components_host.cpp).
//
// Invariant: parent[v] < v for every non-root v, and parent[v] == v for a root.  Every store keeps it: a hook writes
// a smaller root lo under a root hi > lo, and path halving writes a grandparent, which is smaller still.  So
//   * every find terminates, after at most v steps, since each step moves to a smaller vertex;
//   * no cycle can form;
//   * each root is the minimum of its tree, so the root is the canonical label of the component.
// A stale parent read by a concurrent find is still an ancestor (ancestry never changes once made), so it costs a
// retry at most, never a wrong answer: a hook is an atomicCAS on a root, which fails if the root has been hooked.
#pragma once
#include <cstdint>
#include <vector>

#include "icikt_common.cuh"

namespace icikt {

ICIKT_HD int32_t uf_load(const int32_t* a) {
#ifdef __CUDA_ARCH__
  int32_t v;
  asm volatile("ld.relaxed.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(a) : "memory");
  return v;
#else
  return *a;
#endif
}

ICIKT_HD void uf_store(int32_t* a, int32_t v) {
#ifdef __CUDA_ARCH__
  asm volatile("st.relaxed.gpu.global.s32 [%0], %1;" ::"l"(a), "r"(v) : "memory");
#else
  *a = v;
#endif
}

// the root of v's tree, with path halving (every vertex on the path is pointed at its grandparent)
ICIKT_HD int32_t uf_find(int32_t* parent, int32_t v) {
  for (;;) {
    const int32_t p = uf_load(parent + v);
    if (p == v) return v;
    const int32_t g = uf_load(parent + p);
    if (g == p) return p;
    uf_store(parent + v, g);
    v = g;
  }
}

// the root of v's tree without writing: for a pass that reads the forest while others may still halve its paths
ICIKT_HD int32_t uf_root(const int32_t* parent, int32_t v) {
  for (int32_t p; (p = uf_load(parent + v)) != v;) v = p;
  return v;
}

// Joins the trees of a and b; true iff this call hooked one root under the other (then the forest has one tree less).
// No warp-synchronous intrinsic may be called here: lanes leave the loop at different times.
ICIKT_HD bool uf_unite(int32_t* parent, int32_t a, int32_t b) {
  a = uf_find(parent, a);
  b = uf_find(parent, b);
  while (a != b) {
    const int32_t lo = a < b ? a : b, hi = a < b ? b : a;
#ifdef __CUDA_ARCH__
    const int32_t old = atomicCAS(parent + hi, hi, lo);
#else
    const int32_t old = parent[hi];
    if (old == hi) parent[hi] = lo;
#endif
    if (old == hi) return true;
    // hi was hooked meanwhile under old < hi: join lo with hi's new root
    a = lo;
    b = uf_find(parent, old);
  }
  return false;
}

// The labels of several devices merged on the host.  labels[k] holds device k's labels [T][V] (filter-major, each the
// smallest vertex of its component over the device's own edges); out receives, in the same layout, the labels of the
// union of all devices' edges and n_components[f] (may be null) their number.  Each device's forest is a star per
// component, so uniting every v with labels[k][f V + v] joins exactly what the device's edges join.  The labels are
// therefore those one device would have computed over all edges.
inline void merge_component_labels(int T, int64_t V, const std::vector<const int32_t*>& labels, int32_t* out,
                                   int64_t* n_components) {
  for (int f = 0; f < T; ++f) {
    int32_t* parent = out + (int64_t)f * V;
    for (int64_t v = 0; v < V; ++v) parent[v] = (int32_t)v;
    for (const int32_t* l : labels)
      for (int64_t v = 0; v < V; ++v) uf_unite(parent, (int32_t)v, l[(int64_t)f * V + v]);
    // parent[v] < v: in ascending order parent[v] already points at its root
    int64_t roots = 0;
    for (int64_t v = 0; v < V; ++v) {
      if (parent[v] == v) ++roots;
      else parent[v] = parent[parent[v]];
    }
    if (n_components) n_components[f] = roots;
  }
}

}  // namespace icikt
