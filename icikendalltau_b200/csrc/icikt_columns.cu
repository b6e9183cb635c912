// icikt_columns.cu -- K1: per-column preprocessing, done once per column instead of twice per
// pair as in the reference.
//
//   keys                setup_missing_matrix (R/utils.R:1-23) + the NA -> "below the minimum"
//                       substitution of src/kendallc.cpp:214-219, expressed as a sort key:
//                       missing rows get key 0, every other value an order-preserving 64-bit
//                       image of the double (-0.0 == +0.0, as compare_self :15-31 sees them).
//   sort                sortedIndex (src/kendallc.cpp:6-12): a CTA-wide LSD radix ARGSORT written
//                       here (radix_pass below): 4-bit digits, the rows' keys stay where they are
//                       and only the 16-bit row ids move; every thread counts the digits of its own
//                       contiguous slice of the current order in byte counters, one flat scan over
//                       the [digit][thread] counters makes the pass stable.  Stability itself is
//                       irrelevant downstream (rows of a tie group are interchangeable for every
//                       count) but is what makes LSD passes compose.  The passes run on the keys' HIGH
//                       32 bits only; neighbours with equal high words are then put in order by their
//                       low words (repair_equal_high_runs), all 64 bits are sorted only if that gives up.
//   ranks and tables    compare_self + cumsum (:15-31, :250-251) -> dense ranks; tie-group
//                       sizes -> count_rank_tie sums (:103-118) in exact int64; the bit masks
//                       and the tied-row list (rows + dense group index) the pair kernel needs.
//   Three shapes: n <= 8192 one fused kernel per column (keys in shared memory, everything else in
//   registers); n <= 22528 sort kernel with the keys' high words and both row-id buffers in
//   shared memory + rank kernel; longer columns the same sort on global (L2-resident) buffers.
#include <algorithm>
#include <cstdlib>

#include "icikt_internal.h"
#include "icikt_count.cuh"

namespace icikt {
namespace {

constexpr int RANK_THREADS = 512;

__device__ __forceinline__ unsigned long long order_key(double v) {
  if (v == 0.0) v = 0.0;  // -0.0 -> +0.0
  const unsigned long long b = (unsigned long long)__double_as_longlong(v);
  return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ double key_value(unsigned long long k) {
  const unsigned long long b = (k >> 63) ? (k & 0x7fffffffffffffffull) : ~k;
  return __longlong_as_double((long long)b);
}

// block-wide exclusive scan of one int per thread; returns the exclusive prefix, sets total
__device__ __forceinline__ int block_scan_excl(int v, int* warp_sums, int& total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int incl = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const int t = __shfl_up_sync(FULL, incl, d);
    if (lane >= d) incl += t;
  }
  if (lane == 31) warp_sums[warp] = incl;
  __syncthreads();
  int ws = (lane < (int)(blockDim.x >> 5)) ? warp_sums[lane] : 0;
  int wincl = ws;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const int t = __shfl_up_sync(FULL, wincl, d);
    if (lane >= d) wincl += t;
  }
  total = __shfl_sync(FULL, wincl, 31);
  const int wexcl = __shfl_sync(FULL, wincl - ws, warp);
  __syncthreads();
  return wexcl + incl - v;
}

__device__ __forceinline__ long long block_sum_ll(long long v, long long* buf) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int d = 16; d >= 1; d >>= 1) v += __shfl_xor_sync(FULL, v, d);
  if (lane == 0) buf[warp] = v;
  __syncthreads();
  long long t = (lane < (int)(blockDim.x >> 5)) ? buf[lane] : 0;
#pragma unroll
  for (int d = 16; d >= 1; d >>= 1) t += __shfl_xor_sync(FULL, t, d);
  __syncthreads();
  return t;
}

// four sums with one pair of barriers; buf holds 4 * 32 values
__device__ __forceinline__ void block_sum_ll4(long long& a, long long& b, long long& c, long long& d, long long* buf) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = (int)(blockDim.x >> 5);
#pragma unroll
  for (int s = 16; s >= 1; s >>= 1) {
    a += __shfl_xor_sync(FULL, a, s);
    b += __shfl_xor_sync(FULL, b, s);
    c += __shfl_xor_sync(FULL, c, s);
    d += __shfl_xor_sync(FULL, d, s);
  }
  if (lane == 0) {
    buf[warp] = a;
    buf[32 + warp] = b;
    buf[64 + warp] = c;
    buf[96 + warp] = d;
  }
  __syncthreads();
  a = lane < nw ? buf[lane] : 0;
  b = lane < nw ? buf[32 + lane] : 0;
  c = lane < nw ? buf[64 + lane] : 0;
  d = lane < nw ? buf[96 + lane] : 0;
#pragma unroll
  for (int s = 16; s >= 1; s >>= 1) {
    a += __shfl_xor_sync(FULL, a, s);
    b += __shfl_xor_sync(FULL, b, s);
    c += __shfl_xor_sync(FULL, c, s);
    d += __shfl_xor_sync(FULL, d, s);
  }
  __syncthreads();
}

// ---- CTA-wide LSD radix argsort (sortedIndex, src/kendallc.cpp:6-12) ------------------------
// One pass on one 4-bit digit of the keys.  The keys stay in place: `src + (row << stride_shift)`
// addresses the key of a row (shared or global memory, generic loads), `shift` is the digit's bit
// position; `in` is the current order of the 16-bit row ids (nullptr = identity), `out` receives the
// order refined by this digit.  Thread t owns the contiguous positions [t*I, (t+1)*I) of the current
// order (I = ceil(n / T)), so "digit-major, thread-minor, position inside the thread" is the stable
// output order and no warp-level cooperation (match / ballot) is needed:
//   sweep 1  cnt8[d][t]++ for the thread's keys (one byte per digit and thread; the row [d][.] of a
//            warp is 32 consecutive bytes: conflict-free);
//   scan     the counters in memory order ARE the output order: every thread folds 16 consecutive
//            bytes (one 128-bit load), one block scan, 16 exclusive prefixes go to pre16;
//   sweep 2  a key goes to pre16[d][t]++.
// Returns false without writing `out` when every key has the same digit (the order is unchanged):
// count data and other low-entropy columns skip most of their passes.
// cnt8: 16*T bytes, pre16: 16*T u16, misc: 64 words.  I <= 255.
// WIDE (row ids in global memory): a thread's slice is a multiple of 4 ids and is read 8 bytes at a time --
// lanes read at a stride of the slice length, so every 2-byte read would otherwise fetch its own 32-byte sector
// (more ids per load would cost the registers that keep two CTAs on an SM).
template <bool WIDE = false>
__device__ __forceinline__ bool radix_pass(const unsigned char* src, const int stride_shift,
                                           const int shift, const uint16_t* in, uint16_t* out, const int n,
                                           unsigned char* cnt8, uint16_t* pre16, uint32_t* misc, const int T) {
  // T sorting threads (a multiple of 32, <= blockDim.x): a pass costs every thread a fixed ~300
  // instructions on top of ~25 per key, so short columns are sorted by fewer threads with more keys
  // each; the other threads only keep the barriers
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, W = T >> 5;
  const bool on = tid < T;
  const int I = WIDE ? (((n + T - 1) / T + 3) & ~3) : (n + T - 1) / T;
  const int p0 = on ? min(tid * I, n) : n, p1 = min(p0 + I, n);
  const int boff = shift >> 3, bsh = shift & 4;
  // four ids of the current order starting at position p (a multiple of 4); ids behind p1 are not used
  auto ids4 = [&](const int p, uint32_t (&row)[4]) {
    if (!in) {
#pragma unroll
      for (int u = 0; u < 4; ++u) row[u] = (uint32_t)(p + u);
    } else if (p + 4 <= p1) {
      const uint2 v = *reinterpret_cast<const uint2*>(in + p);
      row[0] = v.x & 0xffffu;
      row[1] = v.x >> 16;
      row[2] = v.y & 0xffffu;
      row[3] = v.y >> 16;
    } else {
#pragma unroll
      for (int u = 0; u < 4; ++u) row[u] = (p + u < p1) ? (uint32_t)in[p + u] : 0u;
    }
  };
  if (on) {  // zero this thread's 16 counters' worth of the array (128 bits per thread)
    uint4* z = reinterpret_cast<uint4*>(cnt8);
    z[tid] = make_uint4(0u, 0u, 0u, 0u);
  }
  if (tid == 0) misc[8] = 0u;
  __syncthreads();
  const uint32_t d0 = (src[((size_t)(in ? (uint32_t)in[0] : 0u) << stride_shift) + boff] >> bsh) & 15u;
  bool differs = false;
  unsigned char* mycnt = cnt8 + tid;
  if (WIDE) {
    for (int p = p0; p < p1; p += 4) {
      uint32_t row[4], d[4];
      ids4(p, row);
#pragma unroll
      for (int u = 0; u < 4; ++u)
        d[u] = (p + u < p1) ? (src[((size_t)row[u] << stride_shift) + boff] >> bsh) & 15u : 16u;
#pragma unroll
      for (int u = 0; u < 4; ++u)
        if (d[u] < 16u) {
          differs = differs || d[u] != d0;
          mycnt[d[u] * T] += 1;
        }
    }
  } else
  for (int p = p0; p < p1; p += 4) {
    uint32_t d[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      d[u] = 16u;
      if (p + u < p1) {
        const uint32_t row = in ? (uint32_t)in[p + u] : (uint32_t)(p + u);
        d[u] = (src[((size_t)row << stride_shift) + boff] >> bsh) & 15u;
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u)
      if (d[u] < 16u) {
        differs = differs || d[u] != d0;
        mycnt[d[u] * T] += 1;
      }
  }
  if (__any_sync(FULL, differs) && lane == 0) misc[8] = 1u;
  __syncthreads();
  if (misc[8] == 0u) {  // a single digit value
    __syncthreads();    // misc is rewritten by the next pass
    return false;
  }
  {
    const uint4 c = on ? reinterpret_cast<const uint4*>(cnt8)[tid] : make_uint4(0u, 0u, 0u, 0u);
    const uint32_t w[4] = {c.x, c.y, c.z, c.w};
    uint32_t sum = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const uint32_t h = (w[j] & 0x00ff00ffu) + ((w[j] >> 8) & 0x00ff00ffu);
      sum += (h & 0xffffu) + (h >> 16);
    }
    uint32_t incl = sum;
#pragma unroll
    for (int s2 = 1; s2 < 32; s2 <<= 1) {
      const uint32_t t = __shfl_up_sync(FULL, incl, s2);
      if (lane >= s2) incl += t;
    }
    if (on && lane == 31) misc[16 + warp] = incl;
    __syncthreads();
    const uint32_t wv = lane < W ? misc[16 + lane] : 0u;
    uint32_t wincl = wv;
#pragma unroll
    for (int s2 = 1; s2 < 32; s2 <<= 1) {
      const uint32_t t = __shfl_up_sync(FULL, wincl, s2);
      if (lane >= s2) wincl += t;
    }
    uint32_t run = __shfl_sync(FULL, wincl - wv, warp & 31) + incl - sum;
    uint32_t o[8];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
#pragma unroll
      for (int b = 0; b < 4; b += 2) {
        const uint32_t lo = run;
        run += (w[j] >> (8 * b)) & 0xffu;
        const uint32_t hi = run;
        run += (w[j] >> (8 * b + 8)) & 0xffu;
        o[2 * j + (b >> 1)] = lo | (hi << 16);
      }
    }
    if (on) {
      uint4* pr = reinterpret_cast<uint4*>(pre16) + 2 * tid;
      pr[0] = make_uint4(o[0], o[1], o[2], o[3]);
      pr[1] = make_uint4(o[4], o[5], o[6], o[7]);
    }
  }
  __syncthreads();
  uint16_t* mypre = pre16 + tid;
  if (WIDE) {
    for (int p = p0; p < p1; p += 4) {
      uint32_t row[4], d[4];
      ids4(p, row);
#pragma unroll
      for (int u = 0; u < 4; ++u)
        d[u] = (p + u < p1) ? (src[((size_t)row[u] << stride_shift) + boff] >> bsh) & 15u : 16u;
#pragma unroll
      for (int u = 0; u < 4; ++u)
        if (d[u] < 16u) {
          const uint32_t slot = mypre[d[u] * T];
          mypre[d[u] * T] = (uint16_t)(slot + 1u);
          out[slot] = (uint16_t)row[u];
        }
    }
  } else
  for (int p = p0; p < p1; p += 4) {
    uint32_t d[4], row[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      d[u] = 16u;
      row[u] = 0u;
      if (p + u < p1) {
        row[u] = in ? (uint32_t)in[p + u] : (uint32_t)(p + u);
        d[u] = (src[((size_t)row[u] << stride_shift) + boff] >> bsh) & 15u;
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u)
      if (d[u] < 16u) {
        const uint32_t slot = mypre[d[u] * T];
        mypre[d[u] * T] = (uint16_t)(slot + 1u);
        out[slot] = (uint16_t)row[u];
      }
  }
  __syncthreads();
  return true;
}

// Sorts the rows of one column by the `nbits` key bits starting at bit0 (least significant digit
// first); bufA / bufB ping-pong.  `cur` carries the order between calls (nullptr = identity).
template <bool WIDE = false>
__device__ __forceinline__ const uint16_t* radix_argsort(const unsigned char* src, int stride_shift, int bit0,
                                                         int nbits, const uint16_t* cur, uint16_t* bufA,
                                                         uint16_t* bufB, int n, unsigned char* cnt8,
                                                         uint16_t* pre16, uint32_t* misc, int T) {
  for (int b = bit0; b < bit0 + nbits; b += 4) {
    uint16_t* out = (cur == bufA) ? bufB : bufA;
    if (radix_pass<WIDE>(src, stride_shift, b, cur, out, n, cnt8, pre16, misc, T)) cur = out;
  }
  return cur;
}

// sorting threads for a column of n rows in a CTA of `threads`: about 16 keys per thread
__host__ __device__ inline int sort_threads(int n, int threads) {
  int t = 128;
  while (t < threads && t * 16 < n) t <<= 1;
  return t < threads ? t : threads;
}

// The order by the keys' HIGH 32 bits is almost the order by the keys: two doubles share their high word only
// if they agree to ~6 significant digits (or are integers below 2^21, whose low word is zero anyway).  So the
// sort runs its 8 passes on the high word only and this routine repairs what is left: an odd-even
// transposition restricted to neighbours with EQUAL high words, comparing the low words.  Runs of equal high
// words are short in practice (a few pairs per column of continuous data; tie groups of count data need no
// swap at all), so one or two double rounds suffice.  Returns false if `max_rounds` double rounds did not
// finish the job (long runs of values that differ only in the low word): the caller then sorts all 64 bits.
// Thread t < T owns the pairs (p, p + 1) whose first position lies in its slice; `cur` is read and written.
__device__ __forceinline__ bool repair_equal_high_runs(const unsigned char* hi_src, const int hi_shift, const int hi_off,
                                                       const unsigned char* lo_src, const int lo_shift, const int lo_off,
                                                       uint16_t* cur, const int n, uint32_t* misc, const int T,
                                                       const int max_rounds) {
  const int tid = threadIdx.x;
  const int I = (n + T - 1) / T;
  const int p0 = tid < T ? min(tid * I, n) : n, p1 = min(p0 + I, n);
  for (int round = 0; round < max_rounds; ++round) {
    if (tid == 0) misc[9] = 0u;
    __syncthreads();
    for (int parity = 0; parity < 2; ++parity) {
      bool changed = false;
      for (int p = p0 + ((p0 ^ parity) & 1); p < p1 && p + 1 < n; p += 2) {
        const uint32_t a = cur[p], b = cur[p + 1];
        const uint32_t ha = *reinterpret_cast<const uint32_t*>(hi_src + ((size_t)a << hi_shift) + hi_off);
        const uint32_t hb = *reinterpret_cast<const uint32_t*>(hi_src + ((size_t)b << hi_shift) + hi_off);
        if (ha == hb) {
          const uint32_t la = *reinterpret_cast<const uint32_t*>(lo_src + ((size_t)a << lo_shift) + lo_off);
          const uint32_t lb = *reinterpret_cast<const uint32_t*>(lo_src + ((size_t)b << lo_shift) + lo_off);
          if (la > lb) {
            cur[p] = (uint16_t)b;
            cur[p + 1] = (uint16_t)a;
            changed = true;
          }
        }
      }
      if (changed) misc[9] = 1u;
      __syncthreads();
    }
    const bool done = misc[9] == 0u;
    __syncthreads();  // misc[9] is reset at the top of the next round
    if (done) return true;
  }
  return false;
}

// The same for a column whose keys live in global memory (long columns): the pairs of a parity go to the
// threads round-robin, so the ids are read coalesced, and a row's key is fetched once, all 64 bits.
__device__ __forceinline__ bool repair_equal_high_runs_keys(const unsigned long long* __restrict__ keys, uint16_t* cur,
                                                            const int n, uint32_t* misc, const int max_rounds) {
  const int tid = threadIdx.x, T = blockDim.x;
  for (int round = 0; round < max_rounds; ++round) {
    if (tid == 0) misc[9] = 0u;
    __syncthreads();
    for (int parity = 0; parity < 2; ++parity) {
      bool changed = false;
      for (int p = parity + 2 * tid; p + 1 < n; p += 2 * T) {
        const uint32_t a = cur[p], b = cur[p + 1];
        const unsigned long long ka = keys[a], kb = keys[b];
        if ((uint32_t)(ka >> 32) == (uint32_t)(kb >> 32) && (uint32_t)ka > (uint32_t)kb) {
          cur[p] = (uint16_t)b;
          cur[p + 1] = (uint16_t)a;
          changed = true;
        }
      }
      if (changed) misc[9] = 1u;
      __syncthreads();
    }
    const bool done = misc[9] == 0u;
    __syncthreads();  // misc[9] is reset at the top of the next round
    if (done) return true;
  }
  return false;
}

// the identity order, for a column whose high-word passes were all skipped
__device__ __forceinline__ void fill_identity(uint16_t* buf, int n) {
  for (int t = threadIdx.x; t < n; t += blockDim.x) buf[t] = (uint16_t)t;
  __syncthreads();
}
constexpr int kRepairRounds = 6;

// counters of the sort: cnt8 [16][T] bytes, pre16 [16][T] u16, misc 64 words
__host__ __device__ inline size_t sort_counter_bytes(int threads) { return 48 * (size_t)threads + 256; }

// Short columns (n <= 8192): the WHOLE per-column preprocessing in one kernel, one CTA per
// column, every sorted position held in registers (thread t owns positions t*ITEMS ..).
//   missing marking + order-preserving keys   (64-bit keys parked in shared memory)
//   sort                                      (radix_argsort on the row ids, up to 8 byte passes)
//   dense ranks, tie sums, first-group mask, tied-row list, statistics   (as column_rank_kernel)
// One launch instead of three where the per-column work is a visible share of the whole job.
// Each phase after the sort is one pass over the registers plus one block scan.
template <int SORT_THREADS, int ITEMS>
__global__ void __launch_bounds__(SORT_THREADS)
    column_fused_kernel(const double* __restrict__ data, long long ld, int n, int nstride, int wstride,
                        const double* __restrict__ global_na, int n_global_na, int na_inf,
                        uint16_t* __restrict__ perm, uint16_t* __restrict__ rank, uint16_t* __restrict__ trow,
                        uint16_t* __restrict__ trun, uint16_t* __restrict__ tend, uint32_t* __restrict__ nabits,
                        uint32_t* __restrict__ firstbits, uint16_t* __restrict__ gstart, int gstride,
                        uint16_t* __restrict__ lgrp, ColStats* __restrict__ stats,
                        int32_t* __restrict__ max_tied, uint32_t* __restrict__ tord, const PipeConst pc,
                        const int large_tie, const int direct_budget, const int col0) {
  constexpr int CAP = SORT_THREADS * ITEMS;
  extern __shared__ __align__(16) unsigned char sort_smem[];
  __shared__ int warp_sums[32];
  __shared__ long long llbuf[128];
  __shared__ unsigned long long mnkey;
  __shared__ int n_large;
  __shared__ uint32_t descA[32], descB[32];
  const int col = blockIdx.x + col0, tid = threadIdx.x;
  if (tid == 0) n_large = 0;
  unsigned long long keys[ITEMS];
  uint16_t vals[ITEMS];
  {
    // sort-time layout: [CAP] 64-bit keys by row, two [CAP] row-id buffers, the pass counters
    unsigned long long* skey = reinterpret_cast<unsigned long long*>(sort_smem);
    uint16_t* idA = reinterpret_cast<uint16_t*>(sort_smem + 8 * (size_t)CAP);
    uint16_t* idB = idA + CAP;
    unsigned char* cnt8 = sort_smem + 12 * (size_t)CAP;
    uint16_t* pre16 = reinterpret_cast<uint16_t*>(cnt8 + 16 * SORT_THREADS);
    uint32_t* smisc = reinterpret_cast<uint32_t*>(cnt8 + 48 * SORT_THREADS);
#pragma unroll
    for (int i = 0; i < ITEMS; ++i) {  // striped: a warp reads 32 consecutive rows
      const int r = i * SORT_THREADS + tid;
      bool miss = false;
      if (r < n) {
        const double v = data[(size_t)col * ld + r];
        miss = (v != v) || (na_inf && isinf(v));
        for (int g = 0; g < n_global_na; ++g) miss = miss || (v == global_na[g]);
        skey[r] = miss ? 0ull : order_key(v);
      }
      const uint32_t m = __ballot_sync(FULL, miss);
      if ((tid & 31) == 0 && (r >> 5) < wstride) nabits[(size_t)col * wstride + (r >> 5)] = m;
    }
    __syncthreads();
    const unsigned char* kb = reinterpret_cast<const unsigned char*>(skey);
    const int ts = sort_threads(n, SORT_THREADS);
    const uint16_t* cur = radix_argsort(kb, 3, 32, 32, nullptr, idA, idB, n, cnt8, pre16, smisc, ts);  // high words
    if (!cur) {
      fill_identity(idA, n);
      cur = idA;
    }
    if (!repair_equal_high_runs(kb, 3, 4, kb, 3, 0, const_cast<uint16_t*>(cur), n, smisc, ts, kRepairRounds))
      cur = radix_argsort(kb, 3, 0, 64, nullptr, idA, idB, n, cnt8, pre16, smisc, ts);  // all 64 bits, from scratch
    // blocked arrangement: thread t takes sorted positions t*ITEMS .. (padding sorts last; no value
    // maps to the all-ones key, NaN being missing)
#pragma unroll
    for (int i = 0; i < ITEMS; ++i) {
      const int t = tid * ITEMS + i;
      const uint32_t row = (t < n) ? (cur ? (uint32_t)cur[t] : (uint32_t)t) : 0u;
      vals[i] = (uint16_t)row;
      keys[i] = (t < n) ? skey[row] : ~0ull;
    }
  }
  __syncthreads();  // the sort's shared memory is reused below
  unsigned long long* lastkey = reinterpret_cast<unsigned long long*>(sort_smem);           // [SORT_THREADS]
  uint16_t* gpos = reinterpret_cast<uint16_t*>(sort_smem + 8 * SORT_THREADS);                // [CAP + 2]
  uint32_t* bits = reinterpret_cast<uint32_t*>(sort_smem + 8 * SORT_THREADS + ((2 * (CAP + 2) + 15) & ~15));  // [CAP/32]
  uint32_t* whist = bits + ((CAP / 32 + 3) & ~3);                                            // [CAP]
  const int base = tid * ITEMS;  // blocked arrangement after the sort
  uint16_t* pm = perm + (size_t)col * nstride;
  uint16_t* rk = rank + (size_t)col * nstride;
  const int nwords = (n + 31) >> 5;

  int a_loc = 0;
#pragma unroll
  for (int i = 0; i < ITEMS; ++i) {
    if (base + i < n) pm[base + i] = vals[i];
    a_loc += (keys[i] == 0ull);
  }
  lastkey[tid] = keys[ITEMS - 1];
  int a;
  block_scan_excl(a_loc, warp_sums, a);  // missing rows sort first (key 0)
#pragma unroll
  for (int i = 0; i < ITEMS; ++i)
    if (base + i == a) mnkey = keys[i];
  for (int w = tid; w < nwords; w += SORT_THREADS) bits[w] = 0;
  __syncthreads();
  // NA substitute = min - 0.1 (src/kendallc.cpp:214-219); if that does not move the minimum in
  // fp64 the missing rows tie with it
  bool absorb = false;
  if (a > 0 && a < n) {
    const double mn = key_value(mnkey);
    absorb = (__dsub_rn(mn, 0.1) == mn);
  }
  // group starts (compare_self, :15-31) and dense ranks
  unsigned long long prev = tid > 0 ? lastkey[tid - 1] : 0ull;
  uint32_t fmask = 0;
#pragma unroll
  for (int i = 0; i < ITEMS; ++i) {
    const int t = base + i;
    const bool f = t < n && (t == 0 || (keys[i] != prev && !(t == a && absorb)));
    prev = keys[i];
    fmask |= (uint32_t)f << i;
  }
  int K;
  const int excl = block_scan_excl(__popc(fmask), warp_sums, K);
  {
    int r = excl - 1;
#pragma unroll
    for (int i = 0; i < ITEMS; ++i) {
      const int t = base + i;
      if ((fmask >> i) & 1u) gpos[++r] = (uint16_t)t;
      if (t < n) rk[vals[i]] = (uint16_t)r;
    }
  }
  if (tid == 0) gpos[K] = (uint16_t)n;  // n <= 8192 here
  __syncthreads();
  for (int g = tid; g <= K; g += SORT_THREADS) gstart[(size_t)col * gstride + g] = gpos[g];
  // tie sums over group sizes (count_rank_tie, :103-118), exact int64
  long long s2 = 0, s3 = 0, s5 = 0, ntied = 0, lsq = 0;
  for (int g = tid + 1; g < K; g += SORT_THREADS) {
    const long long t = (long long)gpos[g + 1] - (long long)gpos[g];
    if (t >= large_tie) lsq += t * t;
  }
  lsq = block_sum_ll(lsq, llbuf);
  const int large_from = lsq > (long long)direct_budget * n ? large_tie : 0x7fffffff;
  for (int g = tid; g < K; g += SORT_THREADS) {
    const long long t = (long long)gpos[g + 1] - (long long)gpos[g];
    if (g > 0 && t >= large_from) {  // large tie group: also listed by (start position, size)
      const int k = atomicAdd(&n_large, 1);
      lgrp[(size_t)col * kLargeStride + 2 * k] = gpos[g];
      lgrp[(size_t)col * kLargeStride + 2 * k + 1] = (uint16_t)t;
    }
    if (g > 0 && t > 1) ntied += t;
    if (g == 0 && a > 0) continue;  // the NA group is kept apart for the local perspective
    s2 += t * (t - 1);
    s3 += t * (t - 1) * (t - 2);
    s5 += t * (t - 1) * (2 * t + 5);
  }
  block_sum_ll4(s2, s3, s5, ntied, llbuf);
  const int g0size = (K > 0) ? (int)gpos[1] : 0;
  const int first_run = g0size > 1 ? g0size : 0;
  // membership mask of the first group; rows of the other tied groups with their dense group index
  uint32_t tmask = 0, gmask = 0, lmask = 0;
  int after[ITEMS];  // rows of the item's group from the item to the group's end (tied items only)
  {
    int r = excl - 1;
#pragma unroll
    for (int i = 0; i < ITEMS; ++i) {
      const int t = base + i;
      if ((fmask >> i) & 1u) ++r;
      if (t < first_run) atomicOr(&bits[vals[i] >> 5], 1u << (vals[i] & 31));
      if (t < n && t >= g0size) {
        const int sz = (int)gpos[r + 1] - (int)gpos[r];
        const bool tied = sz > 1;
        tmask |= (uint32_t)tied << i;
        lmask |= (uint32_t)(sz >= large_from) << i;
        after[i] = (int)gpos[r + 1] - t;
        gmask |= (uint32_t)(tied && (int)gpos[r] == t) << i;
      }
    }
  }
  int tot2;
  const int excl2 = block_scan_excl(__popc(tmask) | (__popc(gmask) << 16), warp_sums, tot2);
  {
    int pos = excl2 & 0xffff, gcount = excl2 >> 16;
    uint16_t* tr = trow + (size_t)col * nstride;
    uint16_t* tg = trun + (size_t)col * nstride;
    uint16_t* te = tend + (size_t)col * nstride;
#pragma unroll
    for (int i = 0; i < ITEMS; ++i) {
      if ((gmask >> i) & 1u) ++gcount;
      if ((tmask >> i) & 1u) {
        const bool large = (lmask >> i) & 1u;
        tr[pos] = vals[i];
        tg[pos] = (uint16_t)((gcount - 1) | (large ? kLargeFlag : 0u));
        te[pos] = (uint16_t)(base + i);  // its position in sorted order (the pair kernel's in-place comparison)
        ++pos;
      }
    }
  }
  // ---- walk order for the pair kernel's direct comparison of small tie groups: a tied row is
  // compared with the rows behind it in its group (`walk` of them), so consecutive rows of a group
  // walk t-1, t-2, ... 0 steps and a warp taking them in list order idles half of the time.  Here the
  // tied rows are sorted by walk length, longest first (counting sort), and listed as
  // (list index << 16 | walk): the lanes of a warp then walk equally far.
  if ((tot2 & 0xffff) > 0) {  // block-uniform
    for (int w = tid; w < n; w += SORT_THREADS) whist[w] = 0;
    __syncthreads();
#pragma unroll
    for (int i = 0; i < ITEMS; ++i)
      if ((tmask >> i) & 1u) {
        const uint32_t walk = ((lmask >> i) & 1u) ? 0u : (uint32_t)(after[i] - 1);
        after[i] = (int)(walk | (atomicAdd(&whist[walk], 1u) << 16));  // rank inside the walk class
      }
    __syncthreads();
    {  // class offsets, longest walk first
      const int per = (n + SORT_THREADS - 1) / SORT_THREADS;
      const int hi = n - 1 - tid * per, lo = max(hi - per + 1, 0);
      int sum = 0;
      for (int v = hi; v >= lo; --v) sum += (int)whist[v];
      int total;
      int run = block_scan_excl(sum, warp_sums, total);
      for (int v = hi; v >= lo; --v) {
        const int c = (int)whist[v];
        whist[v] = (uint32_t)run;
        run += c;
      }
    }
    __syncthreads();
    uint32_t* to = tord + (size_t)col * nstride;
    int pos = excl2 & 0xffff;
#pragma unroll
    for (int i = 0; i < ITEMS; ++i)
      if ((tmask >> i) & 1u) {
        const uint32_t walk = (uint32_t)after[i] & 0xffffu;
        to[whist[walk] + ((uint32_t)after[i] >> 16)] = ((uint32_t)pos << 16) | walk;
        ++pos;
      }
  }
  __syncthreads();  // bits complete
  for (int w = tid; w < nwords; w += SORT_THREADS) firstbits[(size_t)col * wstride + w] = bits[w];
  if (tid == 0) {
    ColStats s;
    s.n_na = a;
    s.first_run = first_run;
    s.n_tied = (int)ntied;
    s.n_groups = K;
    int L = 1;
    while ((1 << L) < K) ++L;
    s.levels = L;
    s.g0extra = (a > 0) ? g0size - a : 0;
    s.flags = (absorb ? 1 : 0) | (n_large << 8);
    s.n_tgroups = tot2 >> 16;
    s.s2o = s2;
    s.s3o = s3;
    s.s5o = s5;
    s.cconst = 0;
    stats[col] = s;
    // what the pair kernel's launch tiers are selected by (on the device)
    if (n_large > 0) {
      atomicMax(max_tied + 0, 1);
      atomicMax(max_tied + 1, n_large);
    }
    atomicMax(max_tied + 2, K);
  }
  // ---- cconst: pass A (icikt_count.cuh) over the column's own sorted dense ranks.  They hold no
  // inversion, so what the bucket-free pass counts on them is exactly the per-column constant the
  // pair kernel subtracts.  One 8-key run per thread (kk = 1), two u16 buffers in the shared
  // memory the sort and the tables above no longer need.
  if (K < 2) return;  // constant or all-missing column: cconst stays 0 (block-uniform)
  __syncthreads();    // gpos / bits have been read by everyone
  {
    const int nw = (n + 255) >> 8;  // warps whose 256 positions hold keys; the others only keep the barriers
    const int capc = nw << 8;
    const int L = max(1, 32 - __clz(K - 1));
    const uint32_t bufA = smem_addr(sort_smem), bufB = bufA + 2u * (uint32_t)capc;
    int r = excl - 1;
#pragma unroll
    for (int i = 0; i < ITEMS; ++i) {
      if ((fmask >> i) & 1u) ++r;
      if (base + i < n) Mem<false>::st16(bufA + 2u * (uint32_t)(base + i), (uint32_t)r);
    }
    const uint32_t pad = (1u << L) - 1u;
    for (int q = n + tid; q < capc; q += SORT_THREADS) Mem<false>::st16(bufA + 2u * (uint32_t)q, pad);
    __syncthreads();
    unsigned long long acc = 0;
    if ((tid >> 5) < nw) {
      count_pass<false>(bufA, bufB, 1, nw, L, descA, descB, tid & 31, tid >> 5, pc, acc);
    } else {
      for (int b = count_pass_barriers(L); b > 0; --b) __syncthreads();
    }
    const long long total = block_sum_ll((long long)acc, llbuf);
    if (tid == 0) stats[col].cconst = (uint64_t)total;
  }
}

template <int SORT_THREADS, int ITEMS>
int launch_column_fused(const double* d_data, int64_t ld, const double* d_global_na, int n_global_na, int na_inf,
                        ColumnTables& tab, cudaStream_t stream, int large_tie, int direct_budget, int col0,
                        int ncols) {
  constexpr int CAP = SORT_THREADS * ITEMS;
  const size_t sort_bytes = 12 * (size_t)CAP + sort_counter_bytes(SORT_THREADS);  // keys, two row-id buffers, counters
  const size_t post = 8 * SORT_THREADS + ((2 * (CAP + 2) + 15) & ~15) + 4 * ((CAP / 32 + 3) & ~3) + 4 * (size_t)CAP;
  const size_t pass_a = 2 * 2 * (size_t)SORT_THREADS * 8;  // two u16 buffers of 8 keys per thread
  const size_t smem = std::max(std::max(sort_bytes, post), pass_a);
  const PipeConst pc = make_pipe_const();
  auto kern = column_fused_kernel<SORT_THREADS, ITEMS>;
  // the architectural maximum less the kernel's static shared memory (a fixed value, so that host
  // threads driving different shapes on one device cannot shrink it under each other)
  cudaFuncAttributes fa;
  if (cudaFuncGetAttributes(&fa, kern) != cudaSuccess) return -1;
  if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024 - (int)fa.sharedSizeBytes) != cudaSuccess) return -1;
  kern<<<(unsigned)ncols, SORT_THREADS, smem, stream>>>(d_data, ld, (int)tab.n, (int)tab.nstride, (int)tab.wstride,
                                                        d_global_na, n_global_na, na_inf, tab.perm, tab.rank,
                                                        tab.trow, tab.trun, tab.tend, tab.nabits, tab.firstbits, tab.gstart,
                                                        (int)tab.gstride, tab.lgrp, tab.stats, tab.max_tied, tab.tord, pc, large_tie, direct_budget, col0);
  return launch_status(1);
}

// Long columns (n > 8192): keys + sort in one kernel, one 1024-thread CTA per column.
//   SM = true  (n <= kSortSmemRows): the keys' high words (the low words only if the repair of equal-high
//              runs gives up) and both row-id buffers live in shared memory, 8 bytes per row;
//   SM = false (longer): the row ids ping-pong between `perm` and a scratch column in global memory (L2), the
//              byte of the keys a pair of passes sorts by is staged in shared memory (n bytes).
// Writes the keys by row (keys_in), the sorted order (perm), the keys in sorted order (keys_out, what
// column_rank_kernel walks) and the missing-row bit mask.
constexpr int kSortThreads = 1024;
constexpr int kSortSmemRows = 22528;  // 8 bytes per row + 48 KB of counters within 227 KB
template <bool SM>
__global__ void __launch_bounds__(kSortThreads)
    column_sort_kernel(const double* __restrict__ data, long long ld, int n, int nstride, int wstride,
                       const double* __restrict__ global_na, int n_global_na, int na_inf,
                       unsigned long long* keys_in, unsigned long long* __restrict__ keys_out, uint16_t* perm,
                       uint16_t* vals, uint32_t* __restrict__ nabits, const int col0) {
  extern __shared__ __align__(16) unsigned char sort_smem[];
  const int col = blockIdx.x + col0, tid = threadIdx.x;
  unsigned long long* kin = keys_in + (size_t)col * nstride;
  uint16_t* pm = perm + (size_t)col * nstride;
  uint32_t* part = reinterpret_cast<uint32_t*>(sort_smem);  // SM: [nstride] one half of every key, by row
  uint16_t* idA = SM ? reinterpret_cast<uint16_t*>(sort_smem + 4 * (size_t)nstride) : pm;
  uint16_t* idB = SM ? idA + nstride : vals + (size_t)col * nstride;
  unsigned char* slice = sort_smem;  // !SM: [nstride] the byte of every key the current two passes sort by, by row
  unsigned char* cnt8 = sort_smem + (SM ? 8 * (size_t)nstride : (size_t)nstride);
  uint16_t* pre16 = reinterpret_cast<uint16_t*>(cnt8 + 16 * kSortThreads);
  uint32_t* smisc = reinterpret_cast<uint32_t*>(cnt8 + 48 * kSortThreads);
  const int n32 = (n + 31) & ~31;
  for (int r = tid; r < n32; r += kSortThreads) {  // whole warps: the ballot needs every lane
    bool miss = false;
    if (r < n) {
      const double v = data[(size_t)col * ld + r];
      miss = (v != v) || (na_inf && isinf(v));
      for (int g = 0; g < n_global_na; ++g) miss = miss || (v == global_na[g]);
      const unsigned long long k = miss ? 0ull : order_key(v);
      kin[r] = k;
      if (SM) part[r] = (uint32_t)(k >> 32);
    }
    const uint32_t m = __ballot_sync(FULL, miss);
    if ((tid & 31) == 0 && (r >> 5) < wstride) nabits[(size_t)col * wstride + (r >> 5)] = m;
  }
  __syncthreads();
  // high words first, then the repair of equal-high runs against the low words (read from the key array in
  // global memory: only neighbours with equal high words look there); all 64 bits only if the repair gives up
  const unsigned char* kb = reinterpret_cast<const unsigned char*>(kin);
  const unsigned char* pb = reinterpret_cast<const unsigned char*>(part);
  const uint16_t* cur = nullptr;
  if (SM) {
    cur = radix_argsort(pb, 2, 0, 32, nullptr, idA, idB, n, cnt8, pre16, smisc, kSortThreads);
  } else {
    // long columns: a pass looks up the digit of 60 000 rows in sorted order -- one 32-byte L2 sector per byte
    // if it reads the key array.  The byte the next two passes need is copied to shared memory first (one
    // coalesced sweep over the keys), and the passes read it there.
    for (int byte = 4; byte < 8; ++byte) {
      for (int r = tid; r < n; r += kSortThreads) slice[r] = (unsigned char)(kin[r] >> (8 * byte));
      __syncthreads();
      cur = radix_argsort<true>(slice, 0, 0, 8, cur, idA, idB, n, cnt8, pre16, smisc, kSortThreads);
      __syncthreads();  // the slice is rewritten
    }
  }
  if (!cur) {
    fill_identity(idA, n);
    cur = idA;
  }
  const bool repaired = SM ? repair_equal_high_runs(pb, 2, 0, kb, 3, 0, const_cast<uint16_t*>(cur), n, smisc, kSortThreads, kRepairRounds)
                           : repair_equal_high_runs_keys(kin, const_cast<uint16_t*>(cur), n, smisc, kRepairRounds);
  if (!repaired) {
    if (SM) {
      for (int r = tid; r < n; r += kSortThreads) part[r] = (uint32_t)kin[r];
      __syncthreads();
      cur = radix_argsort(pb, 2, 0, 32, nullptr, idA, idB, n, cnt8, pre16, smisc, kSortThreads);
      __syncthreads();
      for (int r = tid; r < n; r += kSortThreads) part[r] = (uint32_t)(kin[r] >> 32);
      __syncthreads();
      cur = radix_argsort(pb, 2, 0, 32, cur, idA, idB, n, cnt8, pre16, smisc, kSortThreads);
    } else {
      cur = radix_argsort<true>(kb, 3, 0, 64, nullptr, idA, idB, n, cnt8, pre16, smisc, kSortThreads);
    }
  }
  __syncthreads();
  unsigned long long* ko = keys_out + (size_t)col * nstride;
  for (int t = tid; t < n; t += kSortThreads) {
    const uint32_t row = cur ? (uint32_t)cur[t] : (uint32_t)t;
    ko[t] = kin[row];
    if (cur != pm) pm[t] = (uint16_t)row;
  }
}

__global__ void __launch_bounds__(RANK_THREADS)
    column_rank_kernel(const unsigned long long* __restrict__ skeys, int n, int nstride, int wstride,
                       uint16_t* __restrict__ perm, uint16_t* __restrict__ rank,
                       uint16_t* __restrict__ trow, uint16_t* __restrict__ trun, uint16_t* __restrict__ tend,
                       uint32_t* __restrict__ firstbits,
                       uint32_t* __restrict__ gpos_all, uint16_t* __restrict__ gstart_tab, int gstride,
                       uint16_t* __restrict__ lgrp, ColStats* __restrict__ stats,
                       int32_t* __restrict__ max_tied, uint32_t* __restrict__ tord,
                       uint16_t* __restrict__ wrank_all, const int large_tie, const int direct_budget,
                       const int col0) {
  // rows compared directly walk less than 2048 steps: groups below large_tie (<= 2048) rows, or larger
  // ones whose squares sum to at most direct_budget (<= 63) * n (launch_columns clamps both)
  __shared__ int n_large;
  __shared__ int warp_sums[32];
  __shared__ long long llbuf[128];
  __shared__ uint32_t bits[2048];
  __shared__ uint32_t whist[2048];
  const int col = blockIdx.x + col0;
  const int tid = threadIdx.x;
  const unsigned long long* sk = skeys + (size_t)col * nstride;
  uint16_t* pm = perm + (size_t)col * nstride;
  uint16_t* rk = rank + (size_t)col * nstride;
  uint16_t* tr = trow + (size_t)col * nstride;
  uint16_t* tg = trun + (size_t)col * nstride;
  uint16_t* te = tend + (size_t)col * nstride;
  uint32_t* gpos = gpos_all + (size_t)col * (nstride + 64);
  const int n32 = (n + 31) & ~31;
  const int nwords = n32 >> 5;
  if (tid == 0) n_large = 0;

  // missing rows sort first (key 0)
  long long a_ll = 0;
  for (int t = tid; t < n; t += RANK_THREADS) a_ll += (sk[t] == 0ull);
  const int a = (int)block_sum_ll(a_ll, llbuf);
  // NA substitute = min - 0.1 (src/kendallc.cpp:214-219); if that does not move the minimum in
  // fp64 (|min| huge or -Inf) the missing rows tie with it
  bool absorb = false;
  if (a > 0 && a < n) {
    const double mn = key_value(sk[a]);
    absorb = (__dsub_rn(mn, 0.1) == mn);
  }

  // dense ranks in sorted order
  int carry = 0;
  for (int t0 = 0; t0 < n32; t0 += RANK_THREADS) {
    const int t = t0 + tid;
    int flag = 0;
    if (t < n) flag = (t == 0) || ((sk[t] != sk[t - 1]) && !(t == a && absorb));
    int total;
    const int excl = block_scan_excl(flag, warp_sums, total);
    if (t < n) {
      const int r = carry + excl + flag - 1;
      rk[pm[t]] = (uint16_t)r;
      if (flag) gpos[r] = (uint32_t)t;
    }
    carry += total;
  }
  const int K = carry;
  if (tid == 0) gpos[K] = (uint32_t)n;
  __syncthreads();
  for (int g = tid; g <= K; g += RANK_THREADS) gstart_tab[(size_t)col * gstride + g] = (uint16_t)gpos[g];  // n <= 65535

  // tie sums over group sizes (count_rank_tie, src/kendallc.cpp:103-118), exact int64
  long long s2 = 0, s3 = 0, s5 = 0, ntied = 0, lsq = 0;
  for (int g = tid + 1; g < K; g += RANK_THREADS) {
    const long long t = (long long)gpos[g + 1] - (long long)gpos[g];
    if (t >= large_tie) lsq += t * t;
  }
  lsq = block_sum_ll(lsq, llbuf);
  const long long large_from = lsq > (long long)direct_budget * n ? large_tie : 0x7fffffff;
  for (int g = tid; g < K; g += RANK_THREADS) {
    const long long t = (long long)gpos[g + 1] - (long long)gpos[g];
    if (g > 0 && t >= large_from) {  // large tie group: also listed by (start position, size)
      const int k = atomicAdd(&n_large, 1);
      lgrp[(size_t)col * kLargeStride + 2 * k] = (uint16_t)gpos[g];
      lgrp[(size_t)col * kLargeStride + 2 * k + 1] = (uint16_t)t;
    }
    if (g > 0 && t > 1) ntied += t;
    if (g == 0 && a > 0) continue;  // the NA group is kept apart for the local perspective
    s2 += t * (t - 1);
    s3 += t * (t - 1) * (t - 2);
    s5 += t * (t - 1) * (2 * t + 5);
  }
  block_sum_ll4(s2, s3, s5, ntied, llbuf);
  const int g0size = (K > 0) ? (int)gpos[1] : 0;
  const int first_run = g0size > 1 ? g0size : 0;

  // membership mask of the first group
  for (int w = tid; w < nwords; w += RANK_THREADS) bits[w] = 0;
  __syncthreads();
  for (int t = tid; t < first_run; t += RANK_THREADS) {
    const uint32_t row = pm[t];
    atomicOr(&bits[row >> 5], 1u << (row & 31));
  }
  __syncthreads();
  for (int w = tid; w < nwords; w += RANK_THREADS) firstbits[(size_t)col * wstride + w] = bits[w];

  // rows of the other tied groups, in sorted order, with a dense index of their group
  carry = 0;
  int gcarry = 0;
  for (int t0 = 0; t0 < n32; t0 += RANK_THREADS) {
    const int t = t0 + tid;
    int flag = 0, r = 0, gstart = 0, large = 0, after = 0;
    uint16_t row = 0;
    if (t < n && t >= g0size) {
      row = pm[t];
      r = rk[row];
      const uint32_t sz = gpos[r + 1] - gpos[r];
      flag = sz > 1;
      large = (long long)sz >= large_from;
      after = (int)gpos[r + 1] - t;
      gstart = flag && (gpos[r] == (uint32_t)t);
    }
    int total, gtotal;
    const int excl = block_scan_excl(flag, warp_sums, total);
    const int gincl = block_scan_excl(gstart, warp_sums, gtotal) + gstart;
    if (flag) {
      tr[carry + excl] = row;
      tg[carry + excl] = (uint16_t)((gcarry + gincl - 1) | (large ? kLargeFlag : 0u));
      te[carry + excl] = (uint16_t)(large ? carry + excl : carry + excl + after);
    }
    carry += total;
    gcarry += gtotal;
  }

  // walk order of the tied rows for the pair kernel's direct comparison (see column_fused_kernel):
  // counting sort by walk length, longest first; the rank inside a class is parked in the sort's
  // value buffer, which is free by now
  if (carry > 0) {  // block-uniform
    const int m = carry;
    uint16_t* wr = wrank_all + (size_t)col * nstride;
    uint32_t* to = tord + (size_t)col * nstride;
    for (int w = tid; w < 2048; w += RANK_THREADS) whist[w] = 0;
    __syncthreads();  // also: te[] above was written by other threads
    for (int k = tid; k < m; k += RANK_THREADS) {
      const int e = te[k];
      const int walk = e > k ? e - k - 1 : 0;
      wr[k] = (uint16_t)atomicAdd(&whist[walk], 1u);
    }
    __syncthreads();
    {
      constexpr int PER = 2048 / RANK_THREADS;
      const int hi = 2047 - tid * PER;
      int sum = 0;
#pragma unroll
      for (int q = 0; q < PER; ++q) sum += (int)whist[hi - q];
      int total;
      int run = block_scan_excl(sum, warp_sums, total);
#pragma unroll
      for (int q = 0; q < PER; ++q) {
        const int c = (int)whist[hi - q];
        whist[hi - q] = (uint32_t)run;
        run += c;
      }
    }
    __syncthreads();
    for (int k = tid; k < m; k += RANK_THREADS) {
      const int e = te[k];
      const uint32_t walk = e > k ? (uint32_t)(e - k - 1) : 0u;
      to[whist[walk] + wr[k]] = ((uint32_t)k << 16) | walk;
      // from here on `tend` holds the row's position in sorted order instead (what the pair kernel's in-place
      // comparison of small groups reads): e - k rows of its group lie at and behind it, the group ends at
      // gpos[rank + 1]; rows of large groups are never compared, theirs stays unset
      if (e > k) te[k] = (uint16_t)(gpos[rk[tr[k]] + 1] - (uint32_t)(e - k));
    }
  }

  if (tid == 0) {
    ColStats s;
    s.n_na = a;
    s.first_run = first_run;
    s.n_tied = (int)ntied;
    s.n_groups = K;
    int L = 1;
    while ((1 << L) < K) ++L;
    s.levels = L;
    s.g0extra = (a > 0) ? g0size - a : 0;
    s.flags = (absorb ? 1 : 0) | (n_large << 8);
    s.n_tgroups = gcarry;
    s.s2o = s2;
    s.s3o = s3;
    s.s5o = s5;
    s.cconst = 0;
    stats[col] = s;
    if (n_large > 0) {
      atomicMax(max_tied + 0, 1);
      atomicMax(max_tied + 1, n_large);
    }
    atomicMax(max_tied + 2, K);
  }
}

// tier maxima from the statistics of all columns (what the column kernels raise with atomicMax in a
// full run): [0] any large tie group, [1] most large groups, [2] most distinct values of a column
__global__ void max_tied_kernel(const ColStats* __restrict__ stats, int C, int32_t* __restrict__ max_tied) {
  int nl = 0, k = 0;
  for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < C; c += gridDim.x * blockDim.x) {
    nl = max(nl, stats[c].flags >> 8);
    k = max(k, stats[c].n_groups);
  }
#pragma unroll
  for (int d = 16; d >= 1; d >>= 1) {
    nl = max(nl, __shfl_xor_sync(FULL, nl, d));
    k = max(k, __shfl_xor_sync(FULL, k, d));
  }
  if ((threadIdx.x & 31) == 0) {
    if (nl > 0) {
      atomicMax(max_tied + 0, 1);
      atomicMax(max_tied + 1, nl);
    }
    atomicMax(max_tied + 2, k);
  }
}

}  // namespace

int launch_max_tied(ColumnTables& tab, cudaStream_t stream) {
  if (cudaMemsetAsync(tab.max_tied, 0, 4 * sizeof(int32_t), stream) != cudaSuccess) return -1;
  const int C = (int)tab.C;
  max_tied_kernel<<<std::min(64, (C + 255) / 256), 256, 0, stream>>>(tab.stats, C, tab.max_tied);
  return launch_status(1);
}

bool columns_fused(int64_t n) { return n <= 8192 && !getenv("ICIKT_NO_FUSED_COLUMNS"); }

int launch_columns(const double* d_data, int64_t ld, const double* d_global_na, int n_global_na,
                   int na_inf, ColumnTables& tab, ColumnWork& wk, const TiledShape& sh,
                   unsigned char* scratch, cudaStream_t stream, int64_t col_lo, int64_t col_hi) {
  const int n = (int)tab.n;
  const int col0 = (int)col_lo, C = (int)(col_hi - col_lo);  // the columns of this call
  if (C <= 0) return 0;
  const int nstride = (int)tab.nstride, wstride = (int)tab.wstride;
  int launches = 0;
  // tie-group thresholds (icikt_common.cuh); the environment overrides are for tuning sweeps
  int large_tie = kLargeTie, direct_budget = kDirectBudget;
  // at least ceil(n / 512): a column then has fewer large groups than the lgrp table's 512 slots
  if (const char* e = getenv("ICIKT_LARGE_TIE"))
    large_tie = std::min(2048, std::max(std::max(2, (n + kLargeStride / 2 - 1) / (kLargeStride / 2)), atoi(e)));
  if (const char* e = getenv("ICIKT_DIRECT_BUDGET")) direct_budget = std::min(63, std::max(0, atoi(e)));
  // the bit arrays are written in full (words below n32/32) by the kernels below; the padding
  // words up to wstride were zeroed once when the plan was created
  // short columns: 512 threads (more CTAs per SM when there are many columns), else 1024
  // full runs reset the tier maxima here and the kernels below raise them; a partial run (sharded
  // preprocessing) is followed by launch_max_tied once the statistics of every column are in place
  if (col0 == 0 && C == (int)tab.C && cudaMemsetAsync(tab.max_tied, 0, 4 * sizeof(int32_t), stream) != cudaSuccess) return -1;
  if (columns_fused(n)) {
    int l;
#define ICIKT_FUSED(T, I) \
  l = launch_column_fused<T, I>(d_data, ld, d_global_na, n_global_na, na_inf, tab, stream, large_tie, direct_budget, col0, C)
    if (n <= 512) ICIKT_FUSED(512, 1);
    else if (n <= 1024) ICIKT_FUSED(512, 2);
    else if (n <= 2048) ICIKT_FUSED(512, 4);
    else if (n <= 3072) ICIKT_FUSED(512, 6);
    else if (n <= 4096) ICIKT_FUSED(1024, 4);
    else if (n <= 5120) ICIKT_FUSED(1024, 5);
    else if (n <= 6144) ICIKT_FUSED(1024, 6);
    else ICIKT_FUSED(1024, 8);
#undef ICIKT_FUSED
    if (l < 0) return -1;
    return launches + l;  // the fused kernel computes the pass-A constants itself
  } else {
    const bool sm = n <= kSortSmemRows && !getenv("ICIKT_SORT_GLOBAL");
    const size_t smem = (sm ? 8 * (size_t)nstride : (size_t)nstride) + sort_counter_bytes(kSortThreads);
    if (sm) {
      if (cudaFuncSetAttribute(column_sort_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024) != cudaSuccess) return -1;
      column_sort_kernel<true><<<C, kSortThreads, smem, stream>>>(d_data, ld, n, nstride, wstride, d_global_na, n_global_na,
                                                                 na_inf, wk.keys_in, wk.keys_out, tab.perm, wk.vals_in,
                                                                 tab.nabits, col0);
    } else {
      if (cudaFuncSetAttribute(column_sort_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024) != cudaSuccess) return -1;
      column_sort_kernel<false><<<C, kSortThreads, smem, stream>>>(d_data, ld, n, nstride, wstride, d_global_na,
                                                                  n_global_na, na_inf, wk.keys_in, wk.keys_out, tab.perm,
                                                                  wk.vals_in, tab.nabits, col0);
    }
    ++launches;
    if (cudaGetLastError() != cudaSuccess) return -1;
    column_rank_kernel<<<C, RANK_THREADS, 0, stream>>>(wk.keys_out, n, nstride, wstride, tab.perm, tab.rank,
                                                       tab.trow, tab.trun, tab.tend, tab.firstbits,
                                                       wk.gpos, tab.gstart, (int)tab.gstride, tab.lgrp, tab.stats, tab.max_tied,
                                                       tab.tord, wk.vals_in, large_tie, direct_budget, col0);
    ++launches;
    if (cudaGetLastError() != cudaSuccess) return -1;
  }
  const int cl = launch_column_consts(tab, sh, scratch, stream, col_lo, col_hi);
  if (cl < 0) return -1;
  return launches + cl;
}

}  // namespace icikt
