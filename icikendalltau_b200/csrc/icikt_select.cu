// icikt_select.cu -- the selection of the filtered all-pairs call (icikt_all_pairs_edges): an order-preserving
// compaction of one window of the pair order, deterministic, in three kernels:
//   * edge_count_kernel: one CTA per tile of kEdgeTile slots; a warp ballot of the predicate is one mask word
//     per 32 slots, the popcounts summed over the CTA are the tile's count;
//   * edge_scan_kernel: one CTA, the tile counts -> exclusive offsets in place, and the total;
//   * edge_scatter_kernel: one CTA per tile; a tile's 32 mask words are its slots in pair order, so one warp scan
//     over their popcounts gives every word's offset and a kept slot's rank within its word is a popc of the
//     bits below it.  Tiles without a kept slot stop after reading their 32 words.
// HBM-bound: the count pass reads the status and, only for a bound that is given, raw (8 B) and the p-value
// (8 B); the scatter pass reads 1/8 B of mask per slot and the fields of the kept slots.
// The counting pass of the edge-count calls (edge_tally_kernel) tests T filters per slot in one read of the slot and
// writes nothing but counters: per filter, the pairs that pass and every column's degree.
// The selection of the top-k call (icikt_all_pairs_topk) follows the edge kernels: per-column buckets of the
// candidates that beat a column's k-th entry, merged into the column's sorted list (see launch_topk_select).  Over
// several devices, topk_device_merge_kernel folds the devices' lists of a block of columns into one.
#include "icikt_components.cuh"
#include "icikt_edges.cuh"
#include "icikt_internal.h"
#include "icikt_topk.cuh"

namespace icikt {

namespace {

constexpr unsigned FULL = 0xffffffffu;
constexpr int kSelThreads = 256;
constexpr int kSelRounds = kEdgeTile / kSelThreads;  // slots per thread
static_assert(kEdgeTile / 32 == 32, "a tile's mask words are scanned by one warp");

__device__ __forceinline__ double max_so_far(const unsigned long long* bits) {
  const unsigned long long b = *bits;
  return b ? __longlong_as_double((long long)b) : __longlong_as_double(0x7ff8000000000000LL);
}

__global__ void __launch_bounds__(kSelThreads) edge_count_kernel(const EdgeSelect s) {
  __shared__ unsigned warp_sum[kSelThreads / 32];
  const long long tile = blockIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const double m = s.scale_max ? max_so_far(s.max_taumax_bits) : 1.0;
  const bool use_t = s.min_abs_cor == s.min_abs_cor, use_a = s.max_pvalue == s.max_pvalue;
  unsigned cnt = 0;
#pragma unroll
  for (int k = 0; k < kSelRounds; ++k) {
    const long long slot = tile * kEdgeTile + k * kSelThreads + threadIdx.x;
    bool keep = false;
    if (slot < s.n_slots) {
      const int32_t st = s.status[slot];
      if (st == 0) {
        const double raw = use_t ? s.tau[slot] : 0.0;
        const double pv = use_a ? s.pvalue[slot] : 0.0;
        keep = edge_keep_window(st, raw, pv, s.min_abs_cor, s.max_pvalue, s.scale_max != 0, m);
      }
    }
    const unsigned word = __ballot_sync(FULL, keep);
    if (lane == 0) s.mask[(tile * kEdgeTile + k * kSelThreads) / 32 + warp] = word;
    cnt += __popc(word);
  }
  if (lane == 0) warp_sum[warp] = cnt;
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned t = 0;
#pragma unroll
    for (int w = 0; w < kSelThreads / 32; ++w) t += warp_sum[w];
    s.tile_offset[tile] = t;
  }
}

// exclusive scan of n tile counts in place; one CTA of 1024 threads, each owns a contiguous run of tiles
__global__ void __launch_bounds__(1024) edge_scan_kernel(uint32_t* __restrict__ v, long long n,
                                                         unsigned long long* __restrict__ total) {
  __shared__ unsigned long long warp_tot[32];
  const long long per = (n + 1023) / 1024;
  const long long lo = min(n, per * threadIdx.x), hi = min(n, lo + per);
  unsigned long long sum = 0;
  for (long long k = lo; k < hi; ++k) sum += v[k];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  unsigned long long incl = sum;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const unsigned long long o = __shfl_up_sync(FULL, incl, d);
    if (lane >= d) incl += o;
  }
  if (lane == 31) warp_tot[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    unsigned long long w = warp_tot[lane], wi = w;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const unsigned long long o = __shfl_up_sync(FULL, wi, d);
      if (lane >= d) wi += o;
    }
    warp_tot[lane] = wi - w;  // exclusive over the warps
    if (lane == 31) *total = wi;
  }
  __syncthreads();
  unsigned long long run = warp_tot[warp] + incl - sum;
  for (long long k = lo; k < hi; ++k) {
    const unsigned c = v[k];
    v[k] = (uint32_t)run;
    run += c;
  }
}

// last unit of [a, b) whose first slot is <= slot (units are in slot order and the first one starts at or
// before it)
__device__ __forceinline__ long long unit_of(const PairUnit* __restrict__ units, long long a, long long b,
                                             long long slot) {
  while (b - a > 1) {
    const long long mid = (a + b) >> 1;
    if (units[mid].slot0 <= slot) a = mid; else b = mid;
  }
  return a;
}

__global__ void __launch_bounds__(kSelThreads) edge_scatter_kernel(const EdgeSelect s) {
  __shared__ uint32_t words[32];
  __shared__ uint32_t word_off[32];
  __shared__ long long unit_range[2];
  const long long tile = blockIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (warp == 0) {
    const uint32_t w = s.mask[tile * 32 + lane];
    const unsigned c = __popc(w);
    unsigned incl = c;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const unsigned o = __shfl_up_sync(FULL, incl, d);
      if (lane >= d) incl += o;
    }
    words[lane] = w;
    word_off[lane] = incl - c;
    if (lane == 31) unit_range[0] = incl;  // the tile's count, for the early exit
  }
  __syncthreads();
  if (unit_range[0] == 0) return;
  __syncthreads();
  if (threadIdx.x < 2) {  // the units that cover the tile: [first, last]
    const long long first_slot = tile * kEdgeTile;
    const long long last_slot = min((long long)s.n_slots, first_slot + kEdgeTile) - 1;
    unit_range[threadIdx.x] = unit_of(s.units, 0, s.n_units, threadIdx.x ? last_slot : first_slot);
  }
  __syncthreads();
  const long long ua = unit_range[0], ub = unit_range[1] + 1;
  const unsigned base = s.tile_offset[tile];
#pragma unroll
  for (int k = 0; k < kSelRounds; ++k) {
    const int m = k * (kSelThreads / 32) + warp;
    const uint32_t w = words[m];
    if (!((w >> lane) & 1u)) continue;
    const long long slot = tile * kEdgeTile + m * 32 + lane;
    const PairUnit u = s.units[unit_of(s.units, ua, ub, slot)];
    EdgeRow r;
    r.i = u.col;
    r.j = u.j0 + (int32_t)(slot - u.slot0);
    r.raw = s.tau[slot];
    r.pvalue = s.pvalue[slot];
    r.taumax = s.taumax[slot];
    r.completeness = s.completeness[slot];
    s.rows[base + word_off[m] + __popc(w & ((1u << lane) - 1u))] = r;
  }
}

// The edge-count calls: one CTA per tile of kEdgeTile slots, every slot read once (status, raw, p-value) and tested
// against all T filters into a T-bit pass mask held in registers.  Work past the mask follows the set bits only: a
// warp whose 32 masks are all zero (few pairs pass) does no more than count its status classes.  For every filter f
// set in some lane, one ballot gives the warp's count (summed per lane in registers, lane f % 32 owns filter f, then
// one shared atomic per lane and one global atomic per CTA and filter); the row endpoint i is shared by the lanes of a
// unit and usually by the whole warp, so the lanes with the same i add their count with one atomic (match_any), and
// the other endpoint j takes one atomic per passing pair and filter.  A diagonal pair (i == j) adds 1 to its column.
// kUnion (the component calls): after the ballots of a round, each lane unites i and j in the forest of every filter
// its pair passes (icikt_components.cuh), in a loop with no warp-synchronous intrinsic, since lanes retry for
// different counts.  A filter already at one component when the CTA starts is skipped: no further edge can change it.
template <bool kUnion>
__global__ void __launch_bounds__(kSelThreads) edge_tally_kernel(const EdgeTally s) {
  __shared__ unsigned cta_pass[kCountFiltersMax];
  __shared__ unsigned cta_status[16];
  __shared__ long long unit_range[2];
  const long long tile = blockIdx.x;
  const int lane = threadIdx.x & 31, T = s.n_filters;
  if (threadIdx.x < kCountFiltersMax) cta_pass[threadIdx.x] = 0;
  if (threadIdx.x < 16) cta_status[threadIdx.x] = 0;
  if (threadIdx.x < 2) {
    const long long first_slot = tile * kEdgeTile;
    const long long last_slot = min((long long)s.n_slots, first_slot + kEdgeTile) - 1;
    unit_range[threadIdx.x] = unit_of(s.units, 0, s.n_units, threadIdx.x ? last_slot : first_slot);
  }
  unsigned long long open = 0;  // kUnion: the filters with more than one component
  if constexpr (kUnion) {
    __shared__ unsigned open_word[2];
    if (threadIdx.x < kCountFiltersMax) {
      const bool more = threadIdx.x < T && s.hooks[threadIdx.x] + 1 < (unsigned long long)s.C;
      const unsigned w = __ballot_sync(FULL, more);
      if (lane == 0) open_word[threadIdx.x >> 5] = w;
    }
    __syncthreads();
    open = ((unsigned long long)open_word[1] << 32) | open_word[0];
  }
  __syncthreads();
  const long long ua = unit_range[0], ub = unit_range[1] + 1;
  unsigned pass_lo = 0, pass_hi = 0;  // this warp's passing pairs of filters lane and lane + 32
#pragma unroll 1
  for (int r = 0; r < kSelRounds; ++r) {
    const long long slot = tile * kEdgeTile + r * kSelThreads + threadIdx.x;
    int32_t st = -1;
    unsigned long long mask = 0;
    if (slot < s.n_slots) {
      st = s.status[slot];
      if (st == 0) {
        const double raw = s.tau[slot], pv = s.pvalue[slot];
        for (int f = 0; f < T; ++f)
          mask |= (unsigned long long)edge_keep_window(0, raw, pv, s.min_abs_cor[f], s.max_pvalue[f], false, 1.0) << f;
      } else {
        atomicAdd(&cta_status[min(st, 15)], 1u);
      }
    }
    const unsigned ok = __ballot_sync(FULL, st == 0);
    if (lane == 0 && ok) atomicAdd(&cta_status[0], (unsigned)__popc(ok));
    const unsigned any_lo = __reduce_or_sync(FULL, (unsigned)mask), any_hi = __reduce_or_sync(FULL, (unsigned)(mask >> 32));
    unsigned long long any = ((unsigned long long)any_hi << 32) | any_lo;
    if (!any) continue;
    int32_t i = -1, j = -1;
    if (mask) {
      const PairUnit u = s.units[unit_of(s.units, ua, ub, slot)];
      i = u.col;
      j = u.j0 + (int32_t)(slot - u.slot0);
    }
    const unsigned peers = __match_any_sync(FULL, i);
    for (; any; any &= any - 1) {
      const int f = __ffsll((long long)any) - 1;
      const bool bit = (mask >> f) & 1ull;
      const unsigned b = __ballot_sync(FULL, bit);
      if (lane == (f & 31)) {
        if (f < 32) pass_lo += __popc(b); else pass_hi += __popc(b);
      }
      if (s.degree && bit) {
        unsigned long long* deg = s.degree + (long long)f * s.C;
        const unsigned grp = b & peers;
        if (lane == __ffs(grp) - 1) atomicAdd(deg + i, (unsigned long long)__popc(grp));
        if (j != i) atomicAdd(deg + j, 1ull);
      }
    }
    if constexpr (kUnion) {
      for (unsigned long long u = i != j ? mask & open : 0; u; u &= u - 1) {
        const int f = __ffsll((long long)u) - 1;
        if (uf_unite(s.parent + (long long)f * s.C, i, j)) atomicAdd(s.hooks + f, 1ull);
      }
    }
  }
  if (pass_lo) atomicAdd(&cta_pass[lane], pass_lo);
  if (pass_hi) atomicAdd(&cta_pass[lane + 32], pass_hi);
  __syncthreads();
  if (threadIdx.x < T && cta_pass[threadIdx.x]) atomicAdd(s.n_pass + threadIdx.x, (unsigned long long)cta_pass[threadIdx.x]);
  if (threadIdx.x < 16 && cta_status[threadIdx.x])
    atomicAdd(s.status_counts + threadIdx.x, (unsigned long long)cta_status[threadIdx.x]);
}

// The forests of the component calls, filter-major [T][C]: every vertex its own root before the first window
__global__ void __launch_bounds__(kSelThreads) component_init_kernel(int32_t* parent, long long n, long long C) {
  const long long k = (long long)blockIdx.x * kSelThreads + threadIdx.x;
  if (k < n) parent[k] = (int32_t)(k % C);
}

// After the last window, every entry becomes its root, the smallest vertex of its component.  The find only reads:
// a path-halving find could write a grandparent over a root another thread has just stored.  The entries still
// change under the reads, but only ever to an ancestor, so every walk ends at the same root.
__global__ void __launch_bounds__(kSelThreads) component_labels_kernel(int32_t* parent, long long n, long long C) {
  const long long k = (long long)blockIdx.x * kSelThreads + threadIdx.x;
  if (k >= n) return;
  int32_t* forest = parent + (k / C) * C;
  const int32_t v = (int32_t)(k % C);
  uf_store(forest + v, uf_root(forest, v));
}

// Top-k: the count pass (kScatter false) and the scatter pass (true) of one tile of kEdgeTile slots.  Both make
// the same decisions, against the thresholds the previous window's merge left.  A unit's pairs share column i,
// so its candidates for i are counted with one atomic per warp and column.  Columns outside [c_lo, c_hi) keep no
// list and take no candidate; ri, rj are the list rows of i and j.
__device__ __forceinline__ bool topk_takes(const TopkCol& t, int k, unsigned long long key, int32_t partner) {
  return t.n < k || topk_before(key, partner, t.key, t.idx);
}

template <bool kScatter>
__global__ void __launch_bounds__(kSelThreads) topk_bucket_kernel(const TopkSelect s) {
  __shared__ long long unit_range[2];
  const long long tile = blockIdx.x;
  const int lane = threadIdx.x & 31;
  if (threadIdx.x < 2) {
    const long long first_slot = tile * kEdgeTile;
    const long long last_slot = min((long long)s.n_slots, first_slot + kEdgeTile) - 1;
    unit_range[threadIdx.x] = unit_of(s.units, 0, s.n_units, threadIdx.x ? last_slot : first_slot);
  }
  __syncthreads();
  const long long ua = unit_range[0], ub = unit_range[1] + 1;
  for (int r = 0; r < kSelRounds; ++r) {
    const long long slot = tile * kEdgeTile + r * kSelThreads + threadIdx.x;
    int32_t i = -1, j = -1, ri = -1, rj = -1;
    bool take_i = false, take_j = false;
    if (slot < s.n_slots && s.status[slot] == 0) {
      const PairUnit u = s.units[unit_of(s.units, ua, ub, slot)];
      i = u.col;
      j = u.j0 + (int32_t)(slot - u.slot0);
      ri = i - (int32_t)s.c_lo;
      rj = j - (int32_t)s.c_lo;
      const uint32_t L = (uint32_t)(s.c_hi - s.c_lo);
      const unsigned long long key = topk_key(s.tau[slot], s.by);
      take_i = (uint32_t)ri < L && topk_takes(s.col[ri], s.k, key, j);
      take_j = (uint32_t)rj < L && topk_takes(s.col[rj], s.k, key, i);
    }
    const unsigned peers = __match_any_sync(FULL, take_i ? i : -1);
    if (take_i) {
      const int leader = __ffs(peers) - 1;
      unsigned at = 0;
      if (lane == leader) at = atomicAdd(&s.col_count[ri], (unsigned)__popc(peers));
      if (kScatter) {
        at = __shfl_sync(peers, at, leader) + __popc(peers & ((1u << lane) - 1u));
        s.cand[at] = make_uint2((unsigned)slot, (unsigned)j);
      }
    }
    if (take_j) {
      const unsigned at = atomicAdd(&s.col_count[rj], 1u);
      if (kScatter) s.cand[at] = make_uint2((unsigned)slot, (unsigned)i);
    }
  }
}

// One CTA per column that keeps a list (c below is its list row): its bucket is taken in chunks that fill a shared array behind the list; candidates that
// cannot beat the list's k-th entry are dropped, the rest are sorted with the list (bitonic) and the first k
// kept.  Then every thread gathers one entry's fields, from the list or from the window, before any is written.
constexpr int kMergeThreads = kTopkMax;
constexpr int kMergeCap = 2 * kTopkMax;
static_assert(kMergeCap - kTopkMax >= kMergeThreads, "a chunk holds at least one candidate per thread");

__global__ void __launch_bounds__(kMergeThreads) topk_merge_kernel(const TopkSelect s) {
  __shared__ unsigned long long key[kMergeCap];
  __shared__ int32_t part[kMergeCap];
  __shared__ int32_t src[kMergeCap];  // >= 0: window slot; < 0: -1 - position in the list
  __shared__ int fill;
  const long long c = blockIdx.x;
  const uint32_t end = s.col_count[c], beg = c ? s.col_count[c - 1] : 0u;
  if (end == beg) return;
  const int k = s.k, tid = threadIdx.x;
  const long long base = c * k;
  int n = s.col[c].n;
  if (tid < n) {
    key[tid] = topk_key(s.raw[base + tid], s.by);
    part[tid] = s.idx[base + tid];
    src[tid] = -1 - tid;
  }
  for (uint32_t o = beg; o < end;) {
    const uint32_t take = min(end - o, (uint32_t)(kMergeCap - n));
    if (tid == 0) fill = n;
    __syncthreads();
    const bool full = n == k;
    const unsigned long long tk = full ? key[k - 1] : 0ull;
    const int32_t ti = full ? part[k - 1] : 0;
    for (uint32_t q = tid; q < take; q += kMergeThreads) {
      const uint2 e = s.cand[o + q];
      const unsigned long long kk = topk_key(s.tau[e.x], s.by);
      if (!full || topk_before(kk, (int32_t)e.y, tk, ti)) {
        const int at = atomicAdd(&fill, 1);
        key[at] = kk;
        part[at] = (int32_t)e.y;
        src[at] = (int32_t)e.x;
      }
    }
    o += take;
    __syncthreads();
    const int m = fill;
    __syncthreads();
    if (m == n) continue;
    int L = 2;
    while (L < m) L <<= 1;
    for (int q = m + tid; q < L; q += kMergeThreads) {  // padding that sorts last
      key[q] = 0ull;
      part[q] = 0x7fffffff;
    }
    __syncthreads();
    for (int size = 2; size <= L; size <<= 1) {
      for (int stride = size >> 1; stride > 0; stride >>= 1) {
        for (int t = tid; t < L / 2; t += kMergeThreads) {
          const int lo = 2 * t - (t & (stride - 1)), hi = lo + stride;
          const bool up = (lo & size) == 0;
          if (topk_before(key[hi], part[hi], key[lo], part[lo]) == up) {
            const unsigned long long tk2 = key[lo];
            key[lo] = key[hi];
            key[hi] = tk2;
            const int32_t tp = part[lo];
            part[lo] = part[hi];
            part[hi] = tp;
            const int32_t ts = src[lo];
            src[lo] = src[hi];
            src[hi] = ts;
          }
        }
        __syncthreads();
      }
    }
    n = min(m, k);
  }
  double raw = 0.0, pv = 0.0, tm = 0.0, comp = 0.0;
  if (tid < n) {
    const int32_t from = src[tid];
    if (from < 0) {
      const long long q = base + (-1 - from);
      raw = s.raw[q];
      pv = s.pv[q];
      tm = s.tm[q];
      comp = s.comp[q];
    } else {
      raw = s.tau[from];
      pv = s.pvalue[from];
      tm = s.taumax[from];
      comp = s.completeness[from];
    }
  }
  __syncthreads();
  if (tid < n) {
    s.idx[base + tid] = part[tid];
    s.raw[base + tid] = raw;
    s.pv[base + tid] = pv;
    s.tm[base + tid] = tm;
    s.comp[base + tid] = comp;
  }
  if (tid == 0) {
    TopkCol t;
    t.n = n;
    t.key = n == k ? key[k - 1] : 0ull;
    t.idx = n == k ? part[k - 1] : 0;
    s.col[c] = t;
  }
}

// One CTA per column of the block, one thread per list position.  The devices' lists fold one at a time into the
// shared accumulator (at most k entries, best first) by merge path: an entry's new position is its index in its own
// list plus its rank in the other (topk_rank), and entries that land at k or beyond drop out.  Partners are disjoint
// across devices, so the positions are distinct.  Each kept entry remembers (device, position) and its fields are
// read from that device once, after the last fold.
__global__ void __launch_bounds__(kTopkMax) topk_device_merge_kernel(const TopkDeviceMerge m) {
  __shared__ unsigned long long akey[kTopkMax], bkey[kTopkMax];
  __shared__ int32_t apart[kTopkMax], bpart[kTopkMax];
  __shared__ int32_t asrc[kTopkMax];  // device * kTopkMax + position in that device's list
  const long long c = m.c_lo + blockIdx.x;
  const int k = m.k, tid = threadIdx.x;
  const long long base = c * k;
  int a = 0;
  for (int d = 0; d < m.n_dev; ++d) {
    const int b = m.col[d][c].n;
    if (b == 0) continue;
    if (tid < b) {
      bkey[tid] = topk_key(m.list[d][base + tid], m.by);
      bpart[tid] = m.idx[d][base + tid];
    }
    __syncthreads();
    int pa = k, pb = k;
    unsigned long long ka = 0ull;
    int32_t ia = 0, sa = 0;
    if (tid < a) {
      ka = akey[tid];
      ia = apart[tid];
      sa = asrc[tid];
      pa = tid + topk_rank(bkey, bpart, b, ka, ia);
    }
    if (tid < b) pb = tid + topk_rank(akey, apart, a, bkey[tid], bpart[tid]);
    const unsigned long long kb = tid < b ? bkey[tid] : 0ull;
    const int32_t ib = tid < b ? bpart[tid] : 0;
    __syncthreads();
    if (pa < k) {
      akey[pa] = ka;
      apart[pa] = ia;
      asrc[pa] = sa;
    }
    if (pb < k) {
      akey[pb] = kb;
      apart[pb] = ib;
      asrc[pb] = d * kTopkMax + tid;
    }
    a = min(a + b, k);
    __syncthreads();
  }
  const long long ck = m.C * k, blk = (m.c_hi - m.c_lo) * k, o = blockIdx.x * (long long)k + tid;
  if (tid < a) {
    const int d = asrc[tid] / kTopkMax;
    const long long q = base + asrc[tid] % kTopkMax;
    const double* l = m.list[d];
    m.out_idx[o] = apart[tid];
    m.out[o] = l[q];
    m.out[blk + o] = l[ck + q];
    m.out[2 * blk + o] = l[2 * ck + q];
    m.out[3 * blk + o] = l[3 * ck + q];
  }
  if (tid == 0) m.n[blockIdx.x] = a;
}

}  // namespace

int launch_topk_device_merge(const TopkDeviceMerge& m, cudaStream_t stream) {
  if (m.c_hi <= m.c_lo) return launch_status(0);
  if (m.n_dev < 1 || m.n_dev > kMaxMatrixDevices || m.k < 1 || m.k > kTopkMax || m.c_hi - m.c_lo > 0x7fffffffLL)
    return launch_refused("top-k device merge: bad arguments");
  const int threads = (m.k + 31) / 32 * 32;
  topk_device_merge_kernel<<<(unsigned)(m.c_hi - m.c_lo), threads, 0, stream>>>(m);
  return launch_status(1);
}

int launch_topk_select(const TopkSelect& s, cudaStream_t stream) {
  if (s.n_slots <= 0) return launch_status(0);
  const long long tiles = (s.n_slots + kEdgeTile - 1) / kEdgeTile;
  const long long L = s.c_hi - s.c_lo;
  if (tiles > 0x7fffffffLL || s.c_lo < 0 || L < 1 || s.c_hi > 0x7fffffffLL || 2 * s.n_slots > 0xffffffffLL)
    return launch_refused("top-k selection: window too large");
  if (cudaMemsetAsync(s.col_count, 0, sizeof(uint32_t) * (size_t)L, stream) != cudaSuccess)
    return launch_refused("top-k selection: clearing the column counts");
  topk_bucket_kernel<false><<<(unsigned)tiles, kSelThreads, 0, stream>>>(s);
  edge_scan_kernel<<<1, 1024, 0, stream>>>(s.col_count, L, s.total);
  topk_bucket_kernel<true><<<(unsigned)tiles, kSelThreads, 0, stream>>>(s);
  topk_merge_kernel<<<(unsigned)L, kMergeThreads, 0, stream>>>(s);
  return launch_status(4);
}

int launch_edge_tally(const EdgeTally& s, cudaStream_t stream) {
  if (s.n_slots <= 0) return launch_status(0);
  const long long tiles = (s.n_slots + kEdgeTile - 1) / kEdgeTile;
  if (tiles > 0x7fffffffLL || s.n_filters < 1 || s.n_filters > kCountFiltersMax || s.C > 0x7fffffffLL)
    return launch_refused("edge tally: bad arguments");
  if (s.parent)
    edge_tally_kernel<true><<<(unsigned)tiles, kSelThreads, 0, stream>>>(s);
  else
    edge_tally_kernel<false><<<(unsigned)tiles, kSelThreads, 0, stream>>>(s);
  return launch_status(1);
}

int launch_component_init(int32_t* parent, int n_filters, int64_t C, cudaStream_t stream) {
  const long long n = (long long)n_filters * C, blocks = (n + kSelThreads - 1) / kSelThreads;
  if (n <= 0 || C > 0x7fffffffLL || blocks > 0x7fffffffLL) return launch_refused("component init: bad arguments");
  component_init_kernel<<<(unsigned)blocks, kSelThreads, 0, stream>>>(parent, n, C);
  return launch_status(1);
}

int launch_component_labels(int32_t* parent, int n_filters, int64_t C, cudaStream_t stream) {
  const long long n = (long long)n_filters * C, blocks = (n + kSelThreads - 1) / kSelThreads;
  if (n <= 0 || C > 0x7fffffffLL || blocks > 0x7fffffffLL) return launch_refused("component labels: bad arguments");
  component_labels_kernel<<<(unsigned)blocks, kSelThreads, 0, stream>>>(parent, n, C);
  return launch_status(1);
}

int launch_edge_select(const EdgeSelect& s, cudaStream_t stream) {
  if (s.n_slots <= 0) {
    cudaMemsetAsync(s.total, 0, sizeof(unsigned long long), stream);
    return launch_status(0);
  }
  const long long tiles = (s.n_slots + kEdgeTile - 1) / kEdgeTile;
  if (tiles > 0x7fffffffLL) return launch_refused("edge selection: window too large");
  edge_count_kernel<<<(unsigned)tiles, kSelThreads, 0, stream>>>(s);
  edge_scan_kernel<<<1, 1024, 0, stream>>>(s.tile_offset, tiles, s.total);
  edge_scatter_kernel<<<(unsigned)tiles, kSelThreads, 0, stream>>>(s);
  return launch_status(3);
}

}  // namespace icikt
