// icikt_pairs.cu -- K2 (pair kernel), K2-naive (one thread per pair) and K3 (fp64 epilogue).
//
// Replaces, for a whole batch of column pairs, the body of ici_kt():
//   src/kendallc.cpp:247-258  two stable argsorts + dense ranks   -> done once per column in K1
//   src/kendallc.cpp:261-267  joint tie runs (compare_both/which_notzero/diff)   -> ntie
//   src/kendallc.cpp:70-100   kendall_discordant (Fenwick tree, int32)           -> dis (int64)
//   src/kendallc.cpp:280-335  tau / tau_max / variance / p-value                  -> K3
//
// Counting scheme (one CTA per pair, all integer, bit-exact):
//   x := the streamed column (its sorted order `perm` defines the positions), y := the
//   staged column (dense ranks in shared memory, one TMA bulk copy per pair).
//   seq[p] = rank_y[perm_x[p]], 16-bit keys (n <= 65 535).
//   dis = #{p<q : x-group(p) != x-group(q), seq[p] > seq[q]}
//       = INV(seq) - sum over x-groups INV(seq restricted to the group)
//   INV is counted by an MSB-first stable partition of the whole sequence (a wavelet-matrix
//   construction) -- NOT the bottom-up merge sort BASELINE.json's north_star sketches; DESIGN.md
//   section 2 states the deviation and why (same counts, fewer instructions per key).
//   Pass A (icikt_count.cuh: count_pass, count_pass_inplace) runs over all n rows, TWO bits per
//   level, lane-sequential: thread t owns a contiguous range of the sequence, counts its keys per
//   digit class with SIMD-in-a-word adds, two packed warp scans give the class offsets, then the
//   thread walks its range with four running slot indices and scatters the keys (STS.U16).  No
//   ballots and no per-key popc.  The low four bits take one count-only level that stores nothing.  Because every row is present, the bucket layout (keys agreeing
//   on the higher bits) and the number of ones before each bucket are properties of column y
//   alone, so the per-bucket offsets collapse into one per-column constant `cconst` (the raw
//   count of y's own sorted sequence, which has no inversions; computed by K1):
//       INV = sum_levels sum_{zero keys} ones_before - cconst.
//   The first x-group (the missing rows, usually the only large tie group) is written into the
//   sequence already ordered by y from a RANK HISTOGRAM (group_hist: 16-bit counters by
//   shared-memory atomics, one block scan, every thread writes `count` copies of its ranks), so it
//   contributes no inversions and its joint ties are sum C(count, 2).  Small tie groups of x are
//   compared directly in K1's walk order (small_groups_direct), large ones are rewritten in place
//   in ascending y order by the same histogram technique (large_groups_sorted).  Pass B
//   (bucket_pass: one-bit levels on the composite key with explicit bucket boundaries, ballot +
//   clz) survives only as tier 2, for columns with very many large groups x distinct values.
//   When y is (nearly) tie-free the first group's histogram shrinks to ONE BIT per rank, set from the
//   membership masks (popc(first_x & missing_y) rows are only counted), see group_hist.
//   Long vectors (global scratch G, or in place IP != 0: y's rank table is not staged) order the
//   work differently: small_groups_inplace compares on the sequence itself after the gather, and
//   large_groups_sorted2 sorts the large groups; in place, staged_gather fills every position
//   through a rank table that passes through the idle counter area in TMA parts, and
//   large_groups_sorted2 sorts the first group together with the large ones.  Those routines exist
//   only in the long-vector instantiations: the same edits in the short-vector kernel cost it 2-3 %
//   through register allocation (profiles/r02_build_variants_ab.txt).
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>

#include "icikt_internal.h"
#include "icikt_count.cuh"

namespace icikt {
thread_local cudaError_t g_launch_error = cudaSuccess;
thread_local const char* g_launch_note = "";
namespace {


// Exclusive scan of the per-warp totals (every warp computes it redundantly from shared
// memory) and, for the bucketed pass, the count at the nearest bucket start that lies in
// an earlier warp's segment (counts are monotone in position, so that is a running max).
template <bool BUCKETS>
__device__ __forceinline__ void cross_warp(const uint32_t* descT, const int32_t* descB, int nwarps,
                                           int lane, int warp, uint32_t& G, uint32_t& total,
                                           int32_t& carry) {
  const uint32_t v = (lane < nwarps) ? descT[lane] : 0u;
  uint32_t incl = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint32_t t = __shfl_up_sync(FULL, incl, d);
    if (lane >= d) incl += t;
  }
  total = __shfl_sync(FULL, incl, 31);
  const uint32_t excl = incl - v;
  G = __shfl_sync(FULL, excl, warp);
  carry = -1;
  if (BUCKETS) {
    const int32_t bl = (lane < nwarps) ? descB[lane] : -1;
    int32_t babs = (bl >= 0 && lane < warp) ? (int32_t)excl + bl : -1;
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) babs = max(babs, __shfl_xor_sync(FULL, babs, d));
    carry = babs;
  }
}

// Pass B: one counting pass with explicit buckets over a sequence of nwarps*kk*32 32-bit keys
// (x tie group << 16 | y rank; positions >= nreal hold all-ones pads).  Every warp owns kk
// consecutive 32-element chunks; kk is uniform over the CTA.  Each level reads buffer `a` and
// scatters into `b` (ping-pong).  Buckets are runs of equal (key >> (s+1)); acc += ones
// preceding inside the bucket; after level 0 one more sweep on the full key adds, for every real
// element, its index inside its run of equal keys to `ties` (the joint ties).
template <bool G>
__device__ __forceinline__ void bucket_pass(typename Mem<G>::ptr a, typename Mem<G>::ptr b, const int kk,
                                            const int nwarps, const int nreal, const int L,
                                            uint32_t* descT, int32_t* descB, const int lane,
                                            const int warp, uint32_t& acc, uint32_t& ties) {
  typedef Mem<G> M;
  const uint32_t base = (uint32_t)(warp * kk) << 5;
  const uint32_t total_len = (uint32_t)(nwarps * kk) << 5;
  const uint32_t lt = lanemask_lt();
  const uint32_t le = lanemask_le();

  for (int s = L - 1; s >= -1; --s) {
    const bool tie_step = (s < 0);  // every element counts as a "one": counts become positions
    uint32_t bitmask = tie_step ? 0u : (1u << s);
    asm volatile("" : "+r"(bitmask));
    const int sh = s + 1;

    uint32_t T = 0;
    int32_t lastB = -1;
    uint32_t carrylast = 0;
    if (base > 0) carrylast = M::ld32(M::add(a, (int32_t)((base - 1) << 2)));
    const uint32_t prevlast = carrylast;
#pragma unroll 2
    for (int c = 0; c < kk; ++c) {
      const uint32_t pos = base + ((uint32_t)c << 5) + lane;
      const uint32_t e = M::ld32(M::add(a, (int32_t)(pos << 2)));
      const bool one = tie_step || ((e & bitmask) != 0u);
      const uint32_t m = __ballot_sync(FULL, one);
      uint32_t prev = __shfl_up_sync(FULL, e, 1);
      if (lane == 0) prev = carrylast;
      const uint32_t bd = __ballot_sync(FULL, (pos == 0u) || (((e ^ prev) >> sh) != 0u));
      carrylast = __shfl_sync(FULL, e, 31);
      if (bd) lastB = (int32_t)(T + __popc(m & below_top(bd)));
      T += __popc(m);
    }
    if (lane == 0) {
      descT[warp] = T;
      descB[warp] = lastB;
    }
    __syncthreads();

    uint32_t Gp, total;
    int32_t carry;
    cross_warp<true>(descT, descB, nwarps, lane, warp, Gp, total, carry);
    const uint32_t Z = total_len - total;

    uint32_t P = Gp;
    carrylast = prevlast;
#pragma unroll 2
    for (int c = 0; c < kk; ++c) {
      const uint32_t pos = base + ((uint32_t)c << 5) + lane;
      const uint32_t e = M::ld32(M::add(a, (int32_t)(pos << 2)));
      const bool one = tie_step || ((e & bitmask) != 0u);
      const uint32_t m = __ballot_sync(FULL, one);
      const uint32_t P1 = P + __popc(m & lt);
      uint32_t prev = __shfl_up_sync(FULL, e, 1);
      if (lane == 0) prev = carrylast;
      const uint32_t bd = __ballot_sync(FULL, (pos == 0u) || (((e ^ prev) >> sh) != 0u));
      carrylast = __shfl_sync(FULL, e, 31);
      const uint32_t seg = bd & le;
      const uint32_t startP = seg ? P + __popc(m & below_top(seg)) : (uint32_t)carry;
      const uint32_t cnt = P1 - startP;
      if (tie_step) {
        if (pos < (uint32_t)nreal) ties += cnt;
      } else if (!one) {
        acc += cnt;
      }
      if (bd) carry = (int32_t)(P + __popc(m & below_top(bd)));
      if (!tie_step) M::st32(M::add(b, (int32_t)((one ? Z + P1 : pos - P1) << 2)), e);
      P += __popc(m);
    }
    if (tie_step) break;
    __syncthreads();  // also protects descT/descB for the next level
    const typename M::ptr t = a;
    a = b;
    b = t;
  }
}


// Pass A for long vectors, IN PLACE: the same two-bit levels as count_pass, but a thread keeps its
// KK runs (8*KK keys) in registers from the counting sweep to the scatter sweep, so the keys can go
// back into the SAME buffer once every thread has read its range (the barrier that publishes the
// warp totals guarantees that).  One u16 buffer instead of two: vectors up to 64 512 rows stay in
// shared memory (2*cap <= 126 KB) instead of falling back to the L2-resident scratch.
template <int KK>
__device__ __forceinline__ void count_pass_inplace(const uint32_t a, const int nwarps, const int L,
                                                   uint32_t* descA, uint32_t* descB, const int lane,
                                                   const int warp, const PipeConst pc, unsigned long long& acc64,
                                                   const uint32_t lead) {
  typedef Mem<false> M;
  const uint32_t tid = ((uint32_t)warp << 5) + (uint32_t)lane;
  constexpr uint32_t R = (uint32_t)KK << 3;
  const uint32_t my_off = tid * (R << 1);
  const uint32_t my_pos = tid * R;
  const uint32_t cap = ((uint32_t)nwarps << 5) * R;
  const uint32_t ra = a + my_off;
  const bool idle = my_pos + R <= lead;  // inside the leading block of zero keys, see count_pass
  for (int s = (L - 1) & ~1; s >= 4; s -= 2) {
    uint32_t w[KK][4];
    uint32_t cl = 0, ch = 0, cb = 0, wm = 0;
    if (idle) {  // (block-divergent, warp-mostly-uniform) nothing to load: every key is zero
#pragma unroll
      for (int c = 0; c < KK; ++c) w[c][0] = w[c][1] = w[c][2] = w[c][3] = 0u;
    } else
#pragma unroll
    for (int c = 0; c < KK; ++c) {
      M::ld128(ra + (c << 4), w[c][0], w[c][1], w[c][2], w[c][3]);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const uint32_t lo = (w[c][j] >> s) & 0x00010001u, hi = (w[c][j] >> (s + 1)) & 0x00010001u;
        cl = M::fadd(cl, lo, pc.one);
        ch = M::fadd(ch, hi, pc.one);
        cb = M::fadd(cb, lo & hi, pc.one);
        wm += hi * (uint32_t)(4 * c + j);  // word index (compile-time): see count_pass
      }
    }
    const LevelCounts lc = fold_counts(cl, ch, cb, wm);
    const uint32_t n1 = lc.n1, n2 = lc.n2, n3 = lc.n3;
    const uint32_t A = n1 | (n2 << 16), B = n3;
    uint32_t inclA = A, inclB = B;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const uint32_t tA = __shfl_up_sync(FULL, inclA, d), tB = __shfl_up_sync(FULL, inclB, d);
      if (lane >= d) {
        inclA += tA;
        inclB += tB;
      }
    }
    if (lane == 31) {
      descA[warp] = inclA;
      descB[warp] = inclB;
    }
    __syncthreads();  // every range is in registers: the buffer may be overwritten
    const uint32_t vA = (lane < nwarps) ? descA[lane] : 0u, vB = (lane < nwarps) ? descB[lane] : 0u;
    const uint32_t totA = __reduce_add_sync(FULL, vA), totB = __reduce_add_sync(FULL, vB);
    const uint32_t exA = __reduce_add_sync(FULL, (lane < warp) ? vA : 0u) + inclA - A;
    const uint32_t exB = __reduce_add_sync(FULL, (lane < warp) ? vB : 0u) + inclB - B;
    const uint32_t e1 = exA & 0xffffu, e2 = exA >> 16, e3 = exB;
    const uint32_t N1 = totA & 0xffffu, N2 = totA >> 16, N3 = totB;
    const uint32_t N0 = cap - N1 - N2 - N3;
    const uint32_t start1 = N0 + e1, start3 = N0 + N1 + N2 + e3;
    uint32_t Q01 = (start1 << 16) | (my_pos - e1 - e2 - e3);
    uint32_t Q23 = (start3 << 16) | (N0 + N1 + e2);
    uint32_t acc2 = 0;
    uint32_t bLl = 1u << s, bHl = 2u << s, bLh = 1u << (s + 16), bHh = 2u << (s + 16);
    asm volatile("" : "+r"(bLl), "+r"(bHl), "+r"(bLh), "+r"(bHh));
    if (!idle) {  // (idle: the block stays where it is)
#pragma unroll
      for (int c = 0; c < KK; ++c) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          M::step4(Q01, Q23, acc2, w[c][j], bLl, bHl, w[c][j], a, pc);
          M::step4(Q01, Q23, acc2, w[c][j], bLh, bHh, M::hi16(w[c][j], pc.c64k), a, pc);
        }
      }
    }
    (void)N3;
    if (!idle) acc64 += (unsigned long long)level_share(lc, R, acc2, e2 + e3, start1, start3, N0, N2);
    __syncthreads();
  }
  // the low nibble, as in count_pass (the sweep writes nothing, so the keys need not stay in registers)
  NibbleCounts nc = {0u, 0u, 0u, 0u, 0u};
  if (!idle) {
#pragma unroll
    for (int c = 0; c < KK; ++c) {
      uint32_t w[4];
      M::ld128(ra + (c << 4), w[0], w[1], w[2], w[3]);
#pragma unroll
      for (int j = 0; j < 4; ++j) nibble_word<false>(nc, w[j]);
    }
  }
  nibble_level<false>(nc, R, idle, lane, warp, a, acc64);
}

// Per-thread sums of the complete-observations mode for one side of a pair (see group_hist).
struct PwSide {
  unsigned long long S = 0;   // sum over the group's rows of (present rows of the other column below it)
  unsigned long long T = 0;   // ties of the group's present rows in the other column, sum C(count, 2)
  unsigned long long s2 = 0, s3 = 0, s5 = 0;  // tie sums of the other column without the group's rows
  uint32_t k = 0;             // distinct values of the other column left without the group's rows
};

// Rank histogram of a group of rows (x's first tie group -- in particular its missing rows) over
// the dense ranks of another column.
//   EMIT: writes the ranks of the `nrows` rows into buf[0, nrows) in ascending order, so that the
//   group contributes no inversions, and returns (summed over the threads) its joint ties with the
//   other column, sum over ranks of C(count, 2).  The sorted sequence is fully described by the
//   histogram, so nothing is moved:
//     1. hist[rank[row]]++ for the rows, 16-bit counters packed two per word, shared-memory atomics
//        (rank 0 -- the rows missing in both columns, by far the fullest counter -- by ballot);
//     2. every thread folds a contiguous range of counters, one block scan gives its output slot;
//     3. it writes `count` copies of each of its ranks; ranks with a long run are parked in a short
//        list and written by the whole CTA.
//   The histogram lives at the top of `buf` (which the gather fills afterwards), above the `keep`
//   slots at the bottom that must survive; if the K counters do not fit there the ranks are
//   processed in several rounds, and if not even 32 fit, in a 16-word spare in shared memory.
//   Cost ~ 8 nrows + 7 K instead of ~ 38 n for an ordered compaction of the other column's sorted
//   order through the group's membership mask.
//   PW (complete-observations mode, kt_fast use = "pairwise.complete.obs"): the same sweep over
//   the counters also yields, from the other column's group-start table, everything needed to
//   take the group's rows out of the pair: see PwSide.  `a_tbl` = missing rows of the other column.
//   GT: the rank table is read from global memory instead of the staged copy.
//   CZ and skip0: the rows with the other column's lowest rank are counted (ties, mini[18]) but not
//   written: the emitted sequence starts with the group's first nonzero rank (see compact_gather).
template <bool G, bool EMIT, bool PW, bool GT, bool CZ = false>
__device__ __forceinline__ uint32_t group_hist(typename Mem<G>::ptr buf, const int cap, const int keep,
                                               const int nrows, const int K,
                                               const uint16_t* __restrict__ rows,
                                               typename Mem<G>::ptr rank_tbl,
                                               const uint16_t* __restrict__ rank_g,
                                               uint32_t* __restrict__ mini, uint32_t* __restrict__ list,
                                               const int list_cap, uint32_t* descT, uint32_t* list_n,
                                               const int nwarps, const uint16_t* __restrict__ gstart,
                                               const int a_tbl, PwSide& pw, const bool try_bits = false,
                                               const uint32_t* __restrict__ grp_bits = nullptr,
                                               const uint32_t* nab_other = nullptr, const int nwords = 0,
                                               const bool skip0 = false) {
  typedef Mem<G> M;
  const bool Z0 = CZ && skip0;  // the lowest rank is not emitted
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, T = blockDim.x;
  int hw = (cap - ((keep + 1) & ~1)) >> 1;         // counter words available above the kept slots
  typename M::ptr hist = M::add(buf, 2 * cap - 4 * hw);
  if (hw < 16) {
    hw = 16;
    hist = M::from_shared(mini);
  }
  if (EMIT && !PW && try_bits && ((K + 31) >> 5) <= hw) {
    // Fast path for the usual case -- apart from the other column's lowest rank (rows missing in both
    // columns, counted by ballot) no two rows of the group share a rank: ONE BIT per rank instead of a
    // counter.  K / 32 words to clear, scan and walk instead of K / 2 (x's 5 000 missing rows over y's
    // 15 000 ranks: 470 words instead of 7 500, three sweeps each).  A rank met twice raises mini[17] and
    // the general path below redoes the group.
    const int bw = (K + 31) >> 5;
    const typename M::ptr bits = hist;
    for (int w = tid; w < bw; w += T) M::st32(M::add(bits, w << 2), 0u);
    if (tid == 0) mini[17] = 0u;
    __syncthreads();
    // The only caller with try_bits passes grp_bits, so the row-list arm below never runs.  It stays because
    // removing it shifts the register allocation of the short-vector kernels: on a B200 (1000 W, 1965 MHz),
    // K2 got 1.1 % faster on the target, config 5 and config 2 but 0.15 % slower on config 1
    // (0.2825 against 0.2821 ms per step, run-to-run spread 0.0001 ms).
    if (grp_bits) {
      // the group's rows from its membership mask instead of its list: the rows that are also missing in the
      // other column (nab_other; most of x's missing rows at correlated missingness) have its lowest rank and
      // are only counted -- one popcount per word -- and only the others look their rank up
      uint32_t zeros = 0;
      bool dup = false;
      for (int i = tid; i < nwords; i += T) {
        const uint32_t g = __ldg(grp_bits + i), nb = nab_other[i];
        zeros += __popc(g & nb);
        uint32_t m = g & ~nb;
        while (m) {
          const uint32_t row = (uint32_t)(i << 5) + (uint32_t)__ffs((int)m) - 1u;
          m &= m - 1u;
          const uint32_t r = GT ? (uint32_t)__ldg(rank_g + row) : M::ld16(M::add(rank_tbl, (int32_t)(row << 1)));
          if (r == 0u) {
            ++zeros;
          } else {
            const uint32_t bit = 1u << (r & 31u);
            dup = dup || (M::atom_or32(M::add(bits, (int32_t)((r >> 5) << 2)), bit) & bit) != 0u;
          }
        }
      }
      zeros = __reduce_add_sync(FULL, zeros);
      if (lane == 0 && zeros) atomicAdd(mini + 18, zeros);
      if (dup) mini[17] = 1u;
    } else {
      const uint4* px8 = reinterpret_cast<const uint4*>(rows);
      const int lim8 = (nrows + 7) >> 3;
      uint32_t zeros = 0;
      bool dup = false;
      for (int q8w = tid & ~31; q8w < lim8; q8w += T) {  // warp-uniform trip count
        const int q8 = q8w + lane;
        uint4 pv = make_uint4(0u, 0u, 0u, 0u);
        if (q8 < lim8) pv = __ldg(px8 + q8);
        const uint32_t pwd[4] = {pv.x, pv.y, pv.z, pv.w};
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const uint32_t row = (j & 1) ? (pwd[j >> 1] >> 16) : (pwd[j >> 1] & 0xffffu);
          uint32_t r = 0xffffffffu;
          if ((q8 << 3) + j < nrows)
            r = GT ? (uint32_t)__ldg(rank_g + row) : M::ld16(M::add(rank_tbl, (int32_t)(row << 1)));
          zeros += __popc(__ballot_sync(FULL, r == 0u));
          if (r - 1u < 0xfffffffeu) {  // a rank other than 0
            const uint32_t bit = 1u << (r & 31u);
            dup = dup || (M::atom_or32(M::add(bits, (int32_t)((r >> 5) << 2)), bit) & bit) != 0u;
          }
        }
      }
      if (lane == 0 && zeros) atomicAdd(mini + 18, zeros);
      if (dup) mini[17] = 1u;
    }
    __syncthreads();
    if (mini[17] == 0u) {
      const uint32_t Z = mini[18];  // rows with the lowest rank lead the sequence
      if (!Z0)
        for (uint32_t q = tid; q < Z; q += T) M::st16(M::add(buf, (int32_t)(q << 1)), 0u);
      const int wpt = (bw + T - 1) / T, w0 = tid * wpt, w1 = min(w0 + wpt, bw);
      uint32_t mine = 0;
      for (int w = w0; w < w1; ++w) mine += __popc(M::ld32(M::add(bits, w << 2)));
      uint32_t incl = mine;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const uint32_t t = __shfl_up_sync(FULL, incl, d);
        if (lane >= d) incl += t;
      }
      if (lane == 31) descT[warp] = incl;
      __syncthreads();
      const uint32_t v = (lane < nwarps) ? descT[lane] : 0u;
      uint32_t pos = (Z0 ? 0u : Z) + __reduce_add_sync(FULL, (lane < warp) ? v : 0u) + incl - mine;
      for (int w = w0; w < w1; ++w) {
        uint32_t m = M::ld32(M::add(bits, w << 2));
        while (m) {
          const uint32_t b = (uint32_t)__ffs((int)m) - 1u;
          m &= m - 1u;
          M::st16(M::add(buf, (int32_t)(pos << 1)), (uint32_t)(w << 5) + b);
          ++pos;
        }
      }
      __syncthreads();  // the bit area is overwritten by the gather
      return tid == 0 ? (uint32_t)(((unsigned long long)Z * (Z - (Z ? 1u : 0u))) >> 1) : 0u;
    }
    if (tid == 0) mini[18] = 0u;  // the general path counts the lowest rank again
    __syncthreads();
  }
  const int kw = (K + 1) >> 1;                     // counter words needed
  if (hw > kw) hw = kw;
  const int wpt = (hw + T - 1) / T;                // words per thread
  const uint32_t r0 = a_tbl > 0 ? 1u : 0u;         // first rank of the other column that is a value
  uint32_t ties = 0, done = 0;                     // done: output slots filled by earlier rounds
  for (int k0 = 0; k0 < K; k0 += 2 * hw) {
    for (int w = tid; w < hw; w += T) M::st32(M::add(hist, w << 2), 0u);
    if (tid == 0) *list_n = 0u;
    __syncthreads();
    {  // 1. histogram of the rows' ranks inside [k0, k0 + 2 hw)
      const uint4* px8 = reinterpret_cast<const uint4*>(rows);
      const uint32_t span = (uint32_t)(2 * hw);
      const int lim8 = (nrows + 7) >> 3;
      uint32_t zeros = 0;
      for (int q8w = tid & ~31; q8w < lim8; q8w += T) {  // warp-uniform trip count
        const int q8 = q8w + lane;
        uint4 pv = make_uint4(0u, 0u, 0u, 0u);
        if (q8 < lim8) pv = __ldg(px8 + q8);  // perm is readable up to nstride (multiple of 64)
        const uint32_t pwd[4] = {pv.x, pv.y, pv.z, pv.w};
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const uint32_t row = (j & 1) ? (pwd[j >> 1] >> 16) : (pwd[j >> 1] & 0xffffu);
          uint32_t r = 0xffffffffu;
          if ((q8 << 3) + j < nrows)
            r = (GT ? (uint32_t)__ldg(rank_g + row) : M::ld16(M::add(rank_tbl, (int32_t)(row << 1)))) - (uint32_t)k0;
          const bool z = (r == 0u);
          zeros += __popc(__ballot_sync(FULL, z));
          if (r < span && !z) M::red_add32(M::add(hist, (int32_t)((r >> 1) << 2)), (r & 1u) ? 0x10000u : 1u);
        }
      }
      if (lane == 0 && zeros) M::red_add32(hist, zeros);
    }
    __syncthreads();
    // rows of the group with the other column's lowest rank: they lead the emitted sequence
    if (EMIT && k0 == 0 && tid == 0) mini[18] = M::ld32(hist) & 0xffffu;
    // 2. rows per thread range, block scan
    const int w0 = tid * wpt, w1 = min(w0 + wpt, hw);
    uint32_t pos = 0, total = 0;
    if (EMIT) {
      uint32_t mine = 0;
      for (int w = w0; w < w1; ++w) {
        uint32_t c = M::ld32(M::add(hist, w << 2));
        if (Z0 && k0 == 0 && w == 0) c &= 0xffff0000u;
        mine += (c & 0xffffu) + (c >> 16);
      }
      uint32_t incl = mine;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const uint32_t t = __shfl_up_sync(FULL, incl, d);
        if (lane >= d) incl += t;
      }
      if (lane == 31) descT[warp] = incl;
      __syncthreads();
      const uint32_t v = (lane < nwarps) ? descT[lane] : 0u;
      total = __reduce_add_sync(FULL, v);
      pos = done + __reduce_add_sync(FULL, (lane < warp) ? v : 0u) + incl - mine;
    }
    // 3. write the runs / sum up
    for (int w = w0; w < w1; ++w) {
      const uint32_t cw = M::ld32(M::add(hist, w << 2));
      if (!PW && cw == 0u) continue;  // empty counters only matter to the complete-observations sums
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const uint32_t c = h ? (cw >> 16) : (cw & 0xffffu);
        const uint32_t r = (uint32_t)k0 + 2u * (uint32_t)w + (uint32_t)h;
        if (PW && r >= r0 && r < (uint32_t)K) {
          const unsigned long long gs = gstart[r], sz = (unsigned long long)gstart[r + 1] - gs;
          const unsigned long long t = sz - c;  // rows of this value left without the group's rows
          pw.S += (unsigned long long)c * (gs - (unsigned long long)a_tbl);
          pw.T += ((unsigned long long)c * (c - (c ? 1u : 0u))) >> 1;
          pw.k += (t > 0);
          if (t > 1) {
            pw.s2 += t * (t - 1);
            pw.s3 += t * (t - 1) * (t - 2);
            pw.s5 += t * (t - 1) * (2 * t + 5);
          }
        }
        if (EMIT) {
          if (Z0 && r == 0u) {
            ties += (c * (c - (c ? 1u : 0u))) >> 1;
            continue;
          }
          if (c == 1u) {
            M::st16(M::add(buf, (int32_t)(pos << 1)), r);
          } else if (c > 1u) {
            ties += (c * (c - 1u)) >> 1;
            uint32_t slot = 0xffffffffu;
            if (c >= 48u) slot = atomicAdd(list_n, 1u);
            if (slot < (uint32_t)list_cap) {
              list[3 * slot + 0] = r;
              list[3 * slot + 1] = pos;
              list[3 * slot + 2] = c;
            } else {
              for (uint32_t j = 0; j < c; ++j) M::st16(M::add(buf, (int32_t)((pos + j) << 1)), r);
            }
          }
          pos += c;
        }
      }
    }
    done += total;
    __syncthreads();
    if (EMIT) {
      const uint32_t nl = min(*list_n, (uint32_t)list_cap);
      for (uint32_t e = 0; e < nl; ++e) {
        const uint32_t r = list[3 * e], off = list[3 * e + 1], c = list[3 * e + 2];
        for (uint32_t j = tid; j < c; j += T) M::st16(M::add(buf, (int32_t)((off + j) << 1)), r);
      }
      __syncthreads();  // the list and the counters are reused by the next round / overwritten by the gather
    }
  }
  return ties;
}

// Small tie groups of x (other than the first; large groups of a column in large-group mode are
// sorted in place instead): the inversions and the joint ties inside each group by direct
// comparison.  `keys` receives the y ranks (u16) of all m tied rows of x in x order; every thread
// takes a row and compares it with the rows behind it in its group.  The rows come in K1's walk
// order -- (list index << 16 | rows behind it), longest walk first -- so that the lanes of a warp
// walk equally far (in list order a group's rows walk t-1, t-2, ... 0 steps and half of the warp
// idles).  One comparison for the usual isolated tie; K1 bounds the total (groups of kLargeTie rows
// or more are only left to this routine while the sum of their size^2 stays below kDirectBudget * n).
// Runs where y's rank table is staged in shared memory (short vectors); small_groups_inplace elsewhere.
__device__ __forceinline__ void small_groups_direct(const uint32_t keys, const int m,
                                                    const uint16_t* __restrict__ trow,
                                                    const uint32_t* __restrict__ tord,
                                                    const uint32_t rank_tbl, uint32_t& inv, uint32_t& ties) {
  typedef Mem<false> M;
  const int tid = threadIdx.x, T = blockDim.x;
  // the first walk-order entry is fetched before the key gather, later ones one step ahead: the
  // global-load latency would otherwise sit between the barrier and the first comparison
  uint32_t e = (tid < m) ? __ldg(tord + tid) : 0u;
  {  // eight rows per thread and step (the list is readable up to nstride, a multiple of 64)
    const uint4* tr8 = reinterpret_cast<const uint4*>(trow);
    for (int t8 = tid; t8 < ((m + 7) >> 3); t8 += T) {
      const uint4 pv = __ldg(tr8 + t8);
      const uint32_t pw[4] = {pv.x, pv.y, pv.z, pv.w};
      uint32_t o[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const uint32_t r0 = pw[j] & 0xffffu, r1 = pw[j] >> 16;
        const bool v0 = (t8 << 3) + 2 * j < m, v1 = (t8 << 3) + 2 * j + 1 < m;  // rows behind m are stale
        const uint32_t k0 = v0 ? M::ld16(M::add(rank_tbl, (int32_t)(r0 << 1))) : 0u;
        const uint32_t k1 = v1 ? M::ld16(M::add(rank_tbl, (int32_t)(r1 << 1))) : 0u;
        o[j] = k0 | (k1 << 16);
      }
      M::st128(M::add(keys, t8 << 4), o[0], o[1], o[2], o[3]);
    }
  }
  __syncthreads();
  for (int i = tid; i < m; i += T) {
    const uint32_t e_next = (i + T < m) ? __ldg(tord + i + T) : 0u;
    const int walk = (int)(e & 0xffffu), k = (int)(e >> 16);
    if (walk == 0) break;  // sorted: nothing but rows without a walk from here on
    // sign bits instead of compare-and-select: (mine - 1 - other) is negative iff other >= mine,
    // (other - mine - 1) iff other <= mine (16-bit keys); one add and one shift-add each
    const uint32_t mine = M::ld16w(M::add(keys, k << 1));
    const uint32_t m1 = mine - 1u, nm = ~mine;
    uint32_t ge = 0, le = 0;
#pragma unroll 4
    for (int j = k + 1; j <= k + walk; ++j) {
      const uint32_t other = M::ld16w(M::add(keys, j << 1));
      ge += (m1 - other) >> 31;
      le += (other + nm) >> 31;
    }
    inv += (uint32_t)walk - ge;        // other < mine
    ties += ge + le - (uint32_t)walk;  // other == mine
    e = e_next;
  }
  __syncthreads();
}

// The same comparison where y's rank table is not staged (long vectors): on the gathered sequence itself,
// after the gather.  The rows of a tie group are consecutive in x order, so the keys of the rows behind a
// row are the ones behind its position (K1's `tend` table: position in sorted order of every list entry);
// no second lookup of the ranks through L2, no copy of the keys.  Large groups and the first group occupy
// other positions.  Ends with a barrier: for L <= 4 pass A starts with its low-nibble level, whose warps
// park their totals over the first keys of their ranges before any barrier, while slower warps would still
// read those keys here.
template <bool G>
__device__ __forceinline__ void small_groups_inplace(typename Mem<G>::ptr seq, const int m,
                                                     const uint32_t* __restrict__ tord,
                                                     const uint16_t* __restrict__ tpos, uint32_t& inv,
                                                     uint32_t& ties) {
  typedef Mem<G> M;
  const int tid = threadIdx.x, T = blockDim.x;
  for (int i = tid; i < m; i += T) {
    const uint32_t e = __ldg(tord + i);
    const int walk = (int)(e & 0xffffu);
    if (walk == 0) break;  // sorted: nothing but rows without a walk from here on
    const int k = (int)__ldg(tpos + (e >> 16));
    const uint32_t mine = M::ld16w(M::add(seq, k << 1));
    const uint32_t m1 = mine - 1u, nm = ~mine;
    uint32_t ge = 0, le = 0;
#pragma unroll 4
    for (int j = k + 1; j <= k + walk; ++j) {
      const uint32_t other = M::ld16w(M::add(seq, j << 1));
      ge += (m1 - other) >> 31;
      le += (other + nm) >> 31;
    }
    inv += (uint32_t)walk - ge;        // other < mine
    ties += ge + le - (uint32_t)walk;  // other == mine
  }
  __syncthreads();
}

// Large tie groups of x (other than the first): their rows' y-ranks, already gathered into the
// sequence in x order, are rewritten in ascending order group by group, so that the groups
// contribute no inversions to pass A.  Same histogram technique as group_hist, several groups per
// round: bin = (group in batch) * K + rank, as many groups per batch as the counter area holds; if
// not even one group's K counters fit, one group at a time in windows of ranks.  Returns (summed
// over the threads) the joint ties inside those groups.  `pre` is a shared array of 256 words;
// `lg` the column's (start, size) table.  Runs where y's rank table is staged in shared memory (short
// vectors); large_groups_sorted2 elsewhere.
// Rows of one bin met by several lanes are added once (match.any + one atomic per distinct bin).  Plain
// shared-memory atomics are 3 % faster on config 4 (27.7 against 28.6 ms), but the different register
// allocation of the whole kernel costs the tie-free target 2.7 % (278.9 against 271.4 ms, same box clocks;
// profiles/r02_match_dedup_ab.txt), so the deduplicating form stays.
__device__ __forceinline__ uint32_t large_groups_sorted(const uint32_t buf, const uint32_t hist, const int hist_words,
                                                        const uint16_t* __restrict__ permX, const uint32_t rank_tbl,
                                                        const int K, const uint16_t* __restrict__ lg, const int nlg,
                                                        uint32_t* __restrict__ pre, uint32_t* __restrict__ list,
                                                        const int list_cap, uint32_t* descT, uint32_t* list_n,
                                                        const int nwarps) {
  typedef Mem<false> M;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, T = blockDim.x;
  const int bins_avail = 2 * hist_words;
  const int gb_max = max(1, min(255, bins_avail / K));  // groups per batch (pre[] holds 256 words)
  const int Kw = min(K, bins_avail);                    // ranks per window (< K only if gb_max == 1)
  uint32_t ties = 0;
  for (int g0 = 0; g0 < nlg; g0 += gb_max) {
    const int nb = min(gb_max, nlg - g0);
    uint32_t done = 0;  // rows of the (single) group written by earlier windows
    for (int k0 = 0; k0 < K; k0 += Kw) {
      const int kw = min(Kw, K - k0);
      const int bins = nb * kw, hw = (bins + 1) >> 1, wpt = (hw + T - 1) / T;
      if (tid == 0) {
        uint32_t acc = 0;
        for (int j = 0; j < nb; ++j) {
          pre[j] = acc;
          acc += lg[2 * (g0 + j) + 1];
        }
        *list_n = 0u;
      }
      for (int w = tid; w < hw; w += T) M::st32(M::add(hist, w << 2), 0u);
      __syncthreads();
      for (int j = 0; j < nb; ++j) {  // 1. histogram; rows of one bin met by several lanes are added once
        const int s0 = lg[2 * (g0 + j)], t = lg[2 * (g0 + j) + 1];
        for (int qw = tid & ~31; qw < t; qw += T) {  // warp-uniform trip count
          const int q = qw + lane;
          uint32_t bin = 0x80000000u | (uint32_t)lane;  // idle lanes: a key of their own
          bool in = false;
          if (q < t) {
            const uint32_t row = permX[s0 + q];
            const uint32_t r = M::ld16(M::add(rank_tbl, (int32_t)(row << 1))) - (uint32_t)k0;
            in = r < (uint32_t)kw;
            if (in) bin = (uint32_t)(j * kw) + r;
          }
          const uint32_t peers = __match_any_sync(FULL, bin);
          if (in && (peers & ((1u << lane) - 1u)) == 0u)
            M::red_add32(M::add(hist, (int32_t)((bin >> 1) << 2)), (uint32_t)__popc(peers) << ((bin & 1u) * 16u));
        }
      }
      __syncthreads();
      // 2. rows per thread range of counters, block scan
      const int w0 = tid * wpt, w1 = min(w0 + wpt, hw);
      uint32_t mine = 0;
      for (int w = w0; w < w1; ++w) {
        const uint32_t c = M::ld32(M::add(hist, w << 2));
        mine += (c & 0xffffu) + (c >> 16);
      }
      uint32_t incl = mine;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const uint32_t t = __shfl_up_sync(FULL, incl, d);
        if (lane >= d) incl += t;
      }
      if (lane == 31) descT[warp] = incl;
      __syncthreads();
      const uint32_t v = (lane < nwarps) ? descT[lane] : 0u;
      const uint32_t total = __reduce_add_sync(FULL, v);
      uint32_t pos = __reduce_add_sync(FULL, (lane < warp) ? v : 0u) + incl - mine;
      // 3. write the runs: rank r of group j goes to start_j + (rows of the batch before it) - (rows of earlier groups)
      int b = 2 * w0;
      int j = b / kw, r = b - j * kw;
      for (int w = w0; w < w1; ++w) {
        const uint32_t cw = M::ld32(M::add(hist, w << 2));
        if (cw == 0u) {  // most counters are empty: a group touches at most as many ranks as it has rows
          b += 2;
          r += 2;
          while (r >= kw) {
            r -= kw;
            ++j;
          }
          continue;
        }
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const uint32_t c = h ? (cw >> 16) : (cw & 0xffffu);
          if (b < bins && c != 0u) {
            const uint32_t dst = (uint32_t)lg[2 * (g0 + j)] + done + (pos - (kw == K ? pre[j] : 0u));
            const uint32_t rank = (uint32_t)(k0 + r);
            if (c == 1u) {
              M::st16(M::add(buf, (int32_t)(dst << 1)), rank);
            } else {
              ties += (c * (c - 1u)) >> 1;
              uint32_t slot = 0xffffffffu;
              if (c >= 48u) slot = atomicAdd(list_n, 1u);
              if (slot < (uint32_t)list_cap) {
                list[3 * slot + 0] = rank;
                list[3 * slot + 1] = dst;
                list[3 * slot + 2] = c;
              } else {
                for (uint32_t k = 0; k < c; ++k) M::st16(M::add(buf, (int32_t)((dst + k) << 1)), rank);
              }
            }
            pos += c;
          }
          ++b;
          if (++r == kw) {
            r = 0;
            ++j;
          }
        }
      }
      done += total;
      __syncthreads();
      const uint32_t nl = min(*list_n, (uint32_t)list_cap);
      for (uint32_t e = 0; e < nl; ++e) {
        const uint32_t r2 = list[3 * e], off = list[3 * e + 1], c = list[3 * e + 2];
        for (uint32_t k = tid; k < c; k += T) M::st16(M::add(buf, (int32_t)((off + k) << 1)), r2);
      }
      __syncthreads();
    }
  }
  return ties;
}

// Second form of large_groups_sorted, used where y's rank table is not staged in shared memory (long vectors:
// the global-scratch and in-place variants).  Same rounds and counters; what differs is everything around them:
//   * with all of y's ranks in one window, a row's rank is read back from the sequence, where the gather has
//     put rank_y[perm_x[s0 + q]] at position s0 + q (nothing of the batch is rewritten before the barrier
//     that ends the histogram), instead of being looked up again through perm_x;
//   * the batch's (start, size) pairs are fetched once by nb threads into shared memory and warp 0 turns them
//     into the output slot of each group's first counter (instead of one thread walking the global table, and
//     a global load per non-empty counter in the emission);
//   * groups of up to kWideGroup rows are histogrammed by ONE warp each (28 warps evaluating the loop header
//     of every small group cost more than the rows themselves), longer ones by the whole CTA;
//   * runs of kListRun (16) keys and more are parked in the list, longer ones in pieces of kRunPiece, and every
//     list entry is written by one warp (the CTA-wide loop spent 28 loop headers per entry).
// `pre` = 256 words of shared memory: [0,128) the packed group table, [128,256) the output slots.
constexpr int kWideGroup = 512, kListRun = 16, kRunPiece = 512;
template <bool G>
__device__ __forceinline__ uint32_t large_groups_sorted2(typename Mem<G>::ptr buf, typename Mem<G>::ptr hist,
                                                         const int hist_words, const uint16_t* __restrict__ permX,
                                                         const uint16_t* __restrict__ rank_g, const int K,
                                                         const uint16_t* __restrict__ lg, const int nlg,
                                                         uint32_t* __restrict__ pre, uint32_t* __restrict__ list,
                                                         const int list_cap, uint32_t* descT, uint32_t* list_n,
                                                         const int nwarps, const int first = 0,
                                                         uint32_t* lead_out = nullptr) {
  // `first` > 0: the first tie group of x (positions [0, first), usually its missing rows) was gathered in x
  // order like everything else and is sorted here as one more group, ahead of the column's large groups; the
  // rows with y's lowest rank (missing in both columns: by far the fullest counter) are counted by ballot and
  // their number goes to *lead_out (the leading zero keys pass A skips)
  typedef Mem<G> M;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, T = blockDim.x;
  const int vfirst = first > 0 ? 1 : 0;
  uint32_t* grp = pre;         // start | size << 16 of the batch's groups (the table's own layout)
  uint32_t* slot0 = pre + 128;  // start - rows of the batch's earlier groups: where the group's first counter writes
  const uint32_t* lg32 = reinterpret_cast<const uint32_t*>(lg);
  const int bins_avail = 2 * hist_words;
  const int gb_max = max(1, min(128, bins_avail / K));  // groups per batch
  const int Kw = min(K, bins_avail);                    // ranks per window (< K only if gb_max == 1)
  uint32_t ties = 0;
  const int ng = nlg + vfirst;
  for (int g0 = 0; g0 < ng; g0 += gb_max) {
    const int nb = min(gb_max, ng - g0);
    uint32_t done = 0;  // rows of the (single) group written by earlier windows
    for (int k0 = 0; k0 < K; k0 += Kw) {
      const int kw = min(Kw, K - k0);
      const int bins = nb * kw, hw = (bins + 1) >> 1, wpt = (hw + T - 1) / T;
      if (tid < nb) grp[tid] = (g0 + tid < vfirst) ? ((uint32_t)first << 16) : __ldg(lg32 + g0 + tid - vfirst);
      if (tid == 0) *list_n = 0u;
      for (int w = tid; w < hw; w += T) M::st32(M::add(hist, w << 2), 0u);
      __syncthreads();
      if (warp == 0) {  // exclusive prefix of the sizes, four groups per lane
        uint32_t sz[4], sum = 0;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int j = 4 * lane + i;
          sz[i] = j < nb ? grp[j] >> 16 : 0u;
          sum += sz[i];
        }
        uint32_t incl = sum;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
          const uint32_t t = __shfl_up_sync(FULL, incl, d);
          if (lane >= d) incl += t;
        }
        uint32_t before = incl - sum;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int j = 4 * lane + i;
          if (j < nb) slot0[j] = (grp[j] & 0xffffu) - (kw == K ? before : 0u);
          before += sz[i];
        }
      }
      // 1. histogram
      auto add_row = [&](const int j, const int s0, const int q) {
        uint32_t r;
        if (kw == K) {  // the gather has put rank_y[perm_x[s0 + q]] there
          r = M::ld16(M::add(buf, (int32_t)((s0 + q) << 1)));
        } else {
          const uint32_t row = permX[s0 + q];
          r = (uint32_t)__ldg(rank_g + row) - (uint32_t)k0;
        }
        if (r < (uint32_t)kw) {
          const uint32_t bin = (uint32_t)(j * kw) + r;
          M::red_add32(M::add(hist, (int32_t)((bin >> 1) << 2)), 1u << ((bin & 1u) * 16u));
        }
      };
      for (int j = 0; j < nb; ++j) {  // long groups: the whole CTA
        const uint32_t g = grp[j];
        const int t = (int)(g >> 16);
        if (t <= kWideGroup) continue;
        if (vfirst && g0 + j == 0 && k0 == 0) {  // the first group: its rank-0 rows by ballot (warp-uniform trips)
          uint32_t zeros = 0;
          for (int qw = tid & ~31; qw < t; qw += T) {
            const int q = qw + lane;
            uint32_t r = 0xffffffffu;
            if (q < t) {
              if (kw == K) {
                r = M::ld16(M::add(buf, (int32_t)(q << 1)));
              } else {
                const uint32_t row = permX[q];
                r = (uint32_t)__ldg(rank_g + row);
              }
            }
            zeros += __popc(__ballot_sync(FULL, r == 0u));
            if (r != 0u && r < (uint32_t)kw) M::red_add32(M::add(hist, (int32_t)((r >> 1) << 2)), 1u << ((r & 1u) * 16u));
          }
          if (lane == 0 && zeros) M::red_add32(hist, zeros);
          continue;
        }
        for (int q = tid; q < t; q += T) add_row(j, (int)(g & 0xffffu), q);
      }
      for (int j = warp; j < nb; j += nwarps) {  // the others: one warp each
        const uint32_t g = grp[j];
        const int t = (int)(g >> 16);
        if (t > kWideGroup) continue;
        for (int q = lane; q < t; q += 32) add_row(j, (int)(g & 0xffffu), q);
      }
      __syncthreads();
      if (vfirst && g0 == 0 && k0 == 0 && tid == 0 && lead_out) *lead_out = M::ld32(hist) & 0xffffu;
      // 2. rows per thread range of counters, block scan
      const int w0 = tid * wpt, w1 = min(w0 + wpt, hw);
      uint32_t mine = 0;
      for (int w = w0; w < w1; ++w) {
        const uint32_t c = M::ld32(M::add(hist, w << 2));
        mine += (c & 0xffffu) + (c >> 16);
      }
      uint32_t incl = mine;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const uint32_t t = __shfl_up_sync(FULL, incl, d);
        if (lane >= d) incl += t;
      }
      if (lane == 31) descT[warp] = incl;
      __syncthreads();
      const uint32_t v = (lane < nwarps) ? descT[lane] : 0u;
      const uint32_t total = __reduce_add_sync(FULL, v);
      uint32_t pos = __reduce_add_sync(FULL, (lane < warp) ? v : 0u) + incl - mine;
      // 3. write the runs: rank r of group j goes to slot0[j] + (rows of the batch before it)
      int b = 2 * w0;
      int j = b / kw, r = b - j * kw;
      for (int w = w0; w < w1; ++w) {
        const uint32_t cw = M::ld32(M::add(hist, w << 2));
        if (cw == 0u) {  // most counters are empty: a group touches at most as many ranks as it has rows
          b += 2;
          r += 2;
          while (r >= kw) {
            r -= kw;
            ++j;
          }
          continue;
        }
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const uint32_t c = h ? (cw >> 16) : (cw & 0xffffu);
          if (b < bins && c != 0u) {
            const uint32_t dst = slot0[j] + done + pos;
            const uint32_t rank = (uint32_t)(k0 + r);
            if (c == 1u) {
              M::st16(M::add(buf, (int32_t)(dst << 1)), rank);
            } else {
              ties += (c * (c - 1u)) >> 1;
              uint32_t left = c, at = dst;
              if (c >= (uint32_t)kListRun) {  // one list entry per piece, written by a warp each below
                const uint32_t pieces = (c + kRunPiece - 1) / kRunPiece;
                const uint32_t first = atomicAdd(list_n, pieces);
                for (uint32_t i = 0; i < pieces && first + i < (uint32_t)list_cap; ++i) {
                  const uint32_t len = min(left, (uint32_t)kRunPiece);
                  list[3 * (first + i) + 0] = rank;
                  list[3 * (first + i) + 1] = at;
                  list[3 * (first + i) + 2] = len;
                  at += len;
                  left -= len;
                }
              }
              for (uint32_t k = 0; k < left; ++k) M::st16(M::add(buf, (int32_t)((at + k) << 1)), rank);  // short, or list full
            }
            pos += c;
          }
          ++b;
          if (++r == kw) {
            r = 0;
            ++j;
          }
        }
      }
      done += total;
      __syncthreads();
      const uint32_t nl = min(*list_n, (uint32_t)list_cap);
      for (uint32_t e = warp; e < nl; e += nwarps) {
        const uint32_t r2 = list[3 * e], off = list[3 * e + 1], c = list[3 * e + 2];
        for (uint32_t k = lane; k < c; k += 32) M::st16(M::add(buf, (int32_t)((off + k) << 1)), r2);
      }
      __syncthreads();  // list, counters and group table are reused by the next round
    }
  }
  return ties;
}

// The gather of the in-place variant, seq[q] = rank_y[perm_x[q]] for ALL positions (the first group too: it is
// sorted afterwards like a large group).  y's rank table does not fit beside the sequence, but the counter
// area of the large groups is idle at this point: the table goes through it in parts of `part_rows` rows (one
// TMA bulk copy each; two parts at 60 000 rows) and every part is one sweep over perm_x that fills in the
// keys of the rows it holds -- shared-memory lookups instead of one 32-byte L2 sector per 2-byte rank.
// Part 0 was requested by the caller (`mbar` has completed for it); the later parts are fetched here.
__device__ __forceinline__ void staged_gather(const uint32_t seq, const uint32_t tbl, const int part_rows,
                                              const uint16_t* __restrict__ permX,
                                              const uint16_t* __restrict__ rankY_g, const int n, const int nstride,
                                              const int cap, const uint32_t padA, const uint32_t mbar,
                                              uint32_t& phase) {
  typedef Mem<false> M;
  const int tid = threadIdx.x, T = blockDim.x;
  const uint4* px8 = reinterpret_cast<const uint4*>(permX);
  for (int base = 0; base < n; base += part_rows) {
    const uint32_t rows = (uint32_t)min(part_rows, nstride - base);
    if (base > 0) {
      __syncthreads();  // every thread is done with the previous part
      if (tid == 0) bulk_g2s(tbl, rankY_g + base, rows * 2u, mbar);
      mbar_wait(mbar, phase);
      phase ^= 1u;
    }
    auto rk = [&](const uint32_t row) -> uint32_t {
      const uint32_t rel = row - (uint32_t)base;
      return rel < rows ? M::ld16(tbl + (rel << 1)) : 0u;
    };
    for (int q8 = tid; q8 < (cap >> 3); q8 += T) {
      const int q0 = q8 << 3;
      uint32_t o[4];
      if (q0 + 8 <= n) {
        const uint4 pv = __ldg(px8 + q8);
        const uint32_t pw[4] = {pv.x, pv.y, pv.z, pv.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) o[j] = rk(pw[j] & 0xffffu) | (rk(pw[j] >> 16) << 16);
      } else {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int qa = q0 + 2 * j, qb = qa + 1;
          const uint32_t lo = (qa < n) ? rk(permX[qa]) : (base == 0 ? padA : 0u);
          const uint32_t hi = (qb < n) ? rk(permX[qb]) : (base == 0 ? padA : 0u);
          o[j] = lo | (hi << 16);
        }
      }
      if (base > 0) {  // the keys of the earlier parts are in place
        uint32_t a0, a1, a2, a3;
        M::ld128(seq + (q0 << 1), a0, a1, a2, a3);
        o[0] |= a0; o[1] |= a1; o[2] |= a2; o[3] |= a3;
      }
      M::st128(seq + (q0 << 1), o[0], o[1], o[2], o[3]);
    }
  }
}

__device__ __forceinline__ unsigned long long warp_sum_u64(unsigned long long v) {
#pragma unroll
  for (int d = 16; d >= 1; d >>= 1) v += __shfl_xor_sync(FULL, v, d);
  return v;
}

struct TiledParams {
  const uint16_t* perm;
  const uint16_t* rank;
  const uint16_t* trow;
  const uint16_t* trun;
  const uint32_t* tord;
  const uint32_t* nabits;
  const uint32_t* firstbits;
  const ColStats* stats;
  const PairUnit* units;
  const int32_t* pj_list;
  PairRaw* raw;
  PairComplete* pw;              // complete-observations mode: per-pair counts on the shared rows
  const uint16_t* gstart;        // [C][gstride] group-start table (complete-observations mode)
  int gstride;
  const uint16_t* lgrp;          // [C][kLargeStride] large tie groups: (start position, size)
  int region_bytes;              // ping-pong region of this launch: 4*cap (light ties) or 8*cap
  unsigned long long* unit_counter;
  unsigned char* scratch;        // global-memory variant: per-CTA ping-pong region
  long long scratch_stride;      // bytes per CTA
  long long n_units;
  int n, n32, nstride, wstride;
  int kk;  // pass A: 8-key runs per thread (odd); a warp covers 8*kk 32-element chunks
  bool radix;  // pass A: radix-16 levels, counter area behind the two sequence buffers (TiledShape::radix)
  // the launch runs only if K1's device-side maxima (any large tie group, most large groups,
  // most distinct values of a column) select its tier: lets the host enqueue the shapes of all
  // tiers back to back without reading anything back
  const int32_t* max_tied;
  int tier;
  long long budget;  // large groups x distinct values above which pass B takes the tied rows
  PipeConst pc;
  const uint16_t* tpos;  // [C][nstride] sorted position of the tied-row list's entries (ColumnTables::tend)
};

// Shared-memory layout of one CTA (all offsets multiples of 16 bytes)
struct Carve {
  unsigned long long* red;  // [32][4]
  long long* unit_slot;
  unsigned char* region_ptr;  // ping-pong region (shared-memory variant)
  uint32_t region;            // its shared-window address
  uint32_t* nabY;
  uint32_t* mini;   // [16] spare histogram words + [1] list length of the first-group emission
  uint32_t* fmask;  // the emission's list of long runs
  uint32_t* descT;
  int32_t* descB;
  __device__ Carve(unsigned char* p, int wstride, int fwords) {
    red = reinterpret_cast<unsigned long long*>(p);
    p += 8 * 32 * 4;
    unit_slot = reinterpret_cast<long long*>(p);
    p += 16;
    descT = reinterpret_cast<uint32_t*>(p);
    p += 4 * 32;
    descB = reinterpret_cast<int32_t*>(p);
    p += 4 * 32;
    nabY = reinterpret_cast<uint32_t*>(p);
    p += 4 * (size_t)wstride;
    mini = reinterpret_cast<uint32_t*>(p);
    p += 4 * 32;
    fmask = reinterpret_cast<uint32_t*>(p);
    p += 4 * (size_t)fwords;
    region_ptr = p;
    region = smem_addr(p);
  }
};

__host__ __device__ inline int fmask_words(int warps, int kk) { return (warps * kk + 3) & ~3; }
inline size_t tiled_smem_bytes(int region_bytes, int wstride, int fwords) {
  return 8 * 32 * 4 + 16 + 256 + 4 * (size_t)wstride + 128 + 4 * (size_t)fwords + (size_t)region_bytes;
}

template <bool G>
__device__ __forceinline__ typename Mem<G>::ptr region_base(const Carve& sm, const TiledParams& p);
template <>
__device__ __forceinline__ uint32_t region_base<false>(const Carve& sm, const TiledParams&) {
  return sm.region;
}
template <>
__device__ __forceinline__ unsigned char* region_base<true>(const Carve&, const TiledParams& p) {
  return p.scratch + (size_t)blockIdx.x * (size_t)p.scratch_stride;
}

// MAXT/MINB only steer the register allocation (occupancy classes); G selects where the
// ping-pong buffers live (shared memory, or an L2-resident global scratch for long vectors).
// sums four per-thread values over the CTA; the totals are valid in thread 0
__device__ __forceinline__ void block_sum4(unsigned long long* red, int nwarps, unsigned long long& a,
                                           unsigned long long& b, unsigned long long& c, unsigned long long& d) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  a = warp_sum_u64(a);
  b = warp_sum_u64(b);
  c = warp_sum_u64(c);
  d = warp_sum_u64(d);
  __syncthreads();
  if (lane == 0) {
    red[warp * 4 + 0] = a;
    red[warp * 4 + 1] = b;
    red[warp * 4 + 2] = c;
    red[warp * 4 + 3] = d;
  }
  __syncthreads();
  if (tid == 0) {
    a = b = c = d = 0;
    for (int w = 0; w < nwarps; ++w) {
      a += red[w * 4 + 0];
      b += red[w * 4 + 1];
      c += red[w * 4 + 2];
      d += red[w * 4 + 3];
    }
  }
}

// The gather of the tier-0 short-vector kernel with y's lowest-rank keys left out (CZ, see DESIGN.md
// section 2): seq'[q] for the x-present rows, i.e. rank_y[perm_x[q]] for q in [f, n) without the zero
// keys, written behind the nonzero keys of x's first group.  A zero key is never the larger element of an
// inversion, so leaving it out loses exactly the nonzero keys before it: the running write position when
// it is met.  That sum goes to `zt` (this thread's share); returns len', the length of seq' (f < n: x has a
// second group).  A round gives every warp 32 CH consecutive 8-key chunks, lane l takes chunks l, l + 32,
// ... of them (coalesced loads; neighbouring lanes write about 8 slots apart, so the 16-bit stores of a
// warp meet at most ~4 to a bank -- with CH consecutive chunks per lane they were 32 CH slots apart, 16 to a
// bank).  The keys stay in registers across the round's one block scan; the chunks' nonzero counts go
// through one warp scan as 16-bit pairs; the two block-scan arrays alternate between rounds.
template <int CH>
__device__ __forceinline__ uint32_t compact_gather(const uint32_t buf, const uint32_t rank_tbl,
                                                   const uint16_t* __restrict__ permX, const int n, const int f,
                                                   const uint32_t* mini18, uint32_t* descT, uint32_t* descB,
                                                   const int nwarps, uint32_t& zt) {
  static_assert(CH % 2 == 0, "chunk counts are scanned in pairs");
  typedef Mem<false> M;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, T = blockDim.x;
  auto rk = [&](uint32_t row) -> uint32_t { return M::ld16(M::add(rank_tbl, (int32_t)(row << 1))); };
  const uint4* px8 = reinterpret_cast<const uint4*>(permX);
  const int c_end = (n + 7) >> 3;
  uint32_t base = 0xffffffffu;  // slots of seq' filled by the first group and earlier rounds
  bool odd = false;
  for (int c0 = f >> 3; c0 < c_end; c0 += CH * T, odd = !odd) {
    const int cw = c0 + warp * 32 * CH + lane;  // this lane's chunk i is cw + 32 i
    uint32_t k[CH][4];  // two keys per word; 0xffff: not a gathered position
    uint32_t cnt[CH / 2] = {};  // nonzero keys of chunks 2m | 2m+1 (16 bits each)
#pragma unroll
    for (int i = 0; i < CH; ++i) {
      const int c = cw + 32 * i, q0 = c << 3;
      if (q0 >= f && q0 + 8 <= n) {
        const uint4 pv = __ldg(px8 + c);
        const uint32_t pw[4] = {pv.x, pv.y, pv.z, pv.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) k[i][j] = rk(pw[j] & 0xffffu) | (rk(pw[j] >> 16) << 16);
      } else {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int qa = q0 + 2 * j, qb = qa + 1;
          const uint32_t lo = (qa >= f && qa < n) ? rk(permX[qa]) : 0xffffu;
          const uint32_t hi = (qb >= f && qb < n) ? rk(permX[qb]) : 0xffffu;
          k[i][j] = lo | (hi << 16);
        }
      }
      uint32_t nz = 0;
#pragma unroll
      for (int j = 0; j < 4; ++j)
        nz += (uint32_t)(((k[i][j] & 0xffffu) - 1u) < 0xfffeu) + (uint32_t)(((k[i][j] >> 16) - 1u) < 0xfffeu);
      cnt[i >> 1] += (i & 1) ? nz << 16 : nz;
    }
    uint32_t incl[CH / 2];
#pragma unroll
    for (int m = 0; m < CH / 2; ++m) incl[m] = cnt[m];
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
#pragma unroll
      for (int m = 0; m < CH / 2; ++m) {
        const uint32_t t = __shfl_up_sync(FULL, incl[m], d);
        if (lane >= d) incl[m] += t;
      }
    }
    // slot of chunk i inside the warp's part: all lanes' earlier chunks + this chunk's earlier lanes
    uint32_t off[CH], wtot = 0;
#pragma unroll
    for (int m = 0; m < CH / 2; ++m) {
      const uint32_t tot = __shfl_sync(FULL, incl[m], 31), ex = incl[m] - cnt[m];
      off[2 * m] = wtot + (ex & 0xffffu);
      wtot += tot & 0xffffu;
      off[2 * m + 1] = wtot + (ex >> 16);
      wtot += tot >> 16;
    }
    uint32_t* desc = odd ? descB : descT;
    if (lane == 31) desc[warp] = wtot;
    __syncthreads();
    if (base == 0xffffffffu) base = (uint32_t)f - *mini18;  // x's first group: f keys, mini[18] of them zero
    const uint32_t v = (lane < nwarps) ? desc[lane] : 0u;
    const uint32_t wbase = base + __reduce_add_sync(FULL, (lane < warp) ? v : 0u);
    base += __reduce_add_sync(FULL, v);
#pragma unroll
    for (int i = 0; i < CH; ++i) {
      uint32_t pos = wbase + off[i];
#pragma unroll
      for (int h = 0; h < 8; ++h) {
        const uint32_t key = (k[i][h >> 1] >> ((h & 1) * 16)) & 0xffffu;
        if (key - 1u < 0xfffeu) {
          M::st16(M::add(buf, (int32_t)(pos << 1)), key);
          ++pos;
        } else if (key == 0u) {
          zt += pos;
        }
      }
    }
  }
  return base;
}

// PW: complete-observations mode (kt_fast use = "pairwise.complete.obs"): besides the global
// counts the kernel takes the rows missing in either column out of the pair, see PairComplete.
// IP: 0, or the compile-time run count KK of the in-place variant for long vectors (one sequence
// buffer, keys in registers across a level, y's rank table read from global memory).
// CZ: tier 0 only -- pass A runs on the sequence without y's lowest-rank keys (compact_gather) for the pairs
// where that takes a whole warp out of its levels.
template <int MAXT, int MINB, bool G, bool PW, int IP = 0, bool CZ = false>
__global__ void __launch_bounds__(MAXT, MINB) pairs_tiled_kernel(const TiledParams p) {
  static_assert(!CZ || (!G && !PW && IP == 0), "the compacted sequence is for the shared-memory two-buffer kernel");
  typedef Mem<G> M;
  constexpr bool RG = G || IP != 0;    // rank table not staged
  constexpr int AQ = IP != 0 ? 2 : 4;  // bytes of the pass-A buffers in units of cap
  // in place: the rank table passes through the counter area in parts, the first group is sorted with the large ones
  constexpr bool STG = IP != 0;
  // pass A's radix-16 levels (TiledParams::radix) are compiled into the roomy register class only: in the tighter
  // ones they spill more, so a radix shape always launches that class (launch_tiled_cls)
  constexpr bool RX = !G && IP == 0 && MAXT == 1024 && MINB == 1;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int T = blockDim.x, nwarps = T >> 5;
  {
    const bool large = p.max_tied[0] != 0;
    const bool costly = (long long)p.max_tied[1] * p.max_tied[2] > p.budget;
    const int turn = !large ? 0 : (costly ? 2 : 1);
    if (turn != p.tier) return;
  }
  const int n = p.n;
  const int nwords = p.n32 >> 5;
  const int kk = p.kk;       // 8-key runs per thread in pass A
  const int kkc = kk << 3;   // 32-element chunks per warp
  const int cap = (nwarps * kkc) << 5;
  Carve sm(smem_raw, p.wstride, fmask_words(nwarps, kkc));
  const typename M::ptr bufA = region_base<G>(sm, p), bufB16 = M::add(bufA, 2 * cap);
  const uint32_t mbar = smem_addr(sm.unit_slot + 1);  // 8 bytes behind the unit slot
  uint32_t tma_phase = 0;
  if ((!RG || STG) && tid == 0) mbar_init(mbar, 1);
  const uint32_t stage_tbl = smem_addr(sm.region_ptr) + (uint32_t)(AQ * cap);  // STG: the counter area
  const int stage_rows = min(p.nstride, ((p.region_bytes - AQ * cap) >> 1) & ~63);
  // (the first __syncthreads of the unit loop publishes the initialised barrier)

  for (;;) {
    if (tid == 0) *sm.unit_slot = (long long)atomicAdd(p.unit_counter, 1ull);
    __syncthreads();
    const long long u = *sm.unit_slot;
    if (u >= p.n_units) break;
    const PairUnit unit = p.units[u];
    const int ycol = unit.col;
    const ColStats YS = p.stats[ycol];
    {  // stage the missing mask of column y (shared by all pairs of the unit)
      const uint32_t* nb = p.nabits + (size_t)ycol * p.wstride;
      for (int i = tid; i < nwords; i += T) sm.nabY[i] = nb[i];
    }
    const uint16_t* rankY_g = p.rank + (size_t)ycol * p.nstride;
    const uint32_t* g0Yg = ((YS.flags & 1) ? p.firstbits : p.nabits) + (size_t)ycol * p.wstride;
    // y's dense-rank table: staged into the second ping-pong buffer, or read in place (RG)
    const typename M::ptr rank_tbl = bufB16;
    const int L = YS.levels;
    const uint32_t padA = (1u << L) - 1u;
    __syncthreads();

    for (int k = 0; k < unit.count; ++k) {
      const long long slot = unit.slot0 + k;
      const int xcol = unit.j_explicit ? p.pj_list[slot] : unit.j0 + k;
      const ColStats XS = p.stats[xcol];
      const uint16_t* permX = p.perm + (size_t)xcol * p.nstride;
      const uint32_t* fbXg = p.firstbits + (size_t)xcol * p.wstride;
      const uint32_t* nbXg = p.nabits + (size_t)xcol * p.wstride;
      const bool absorbed = ((XS.flags | YS.flags) & 1) != 0;
      // y's dense ranks go to the second sequence buffer (free since the barrier that ended the
      // previous pair) as one TMA bulk copy, in flight during the mask counting below
      if (!RG && tid == 0)
        bulk_g2s(smem_addr(sm.region_ptr) + 2u * (uint32_t)cap, rankY_g, (uint32_t)p.nstride * 2u, mbar);
      if (STG && tid == 0)  // first part of y's rank table into the idle counter area
        bulk_g2s(stage_tbl, rankY_g, (uint32_t)min(stage_rows, p.nstride) * 2u, mbar);
      if (tid == 0) sm.mini[18] = 0u;  // leading zero keys of the sequence (set by the first-group emission)
      // joint-missing rows (b) and joint lowest group (g00, differs from b only if a column's
      // missing rows tie with its minimum)
      uint32_t bpart = 0, g00part = 0;
      for (int i = tid; i < nwords; i += T) {
        const uint32_t nb = nbXg[i];
        bpart += __popc(nb & sm.nabY[i]);
        if (absorbed) g00part += __popc(((XS.flags & 1) ? fbXg[i] : nb) & g0Yg[i]);
      }
      if (!RG || STG) {  // the rank table has landed (also on the early exit below: the barrier is reused)
        mbar_wait(mbar, tma_phase);
        tma_phase ^= 1u;
      }
      if (YS.n_groups < 2 || XS.n_groups < 2) {
        // a constant or all-missing column: K3 reports NA; only the joint-missing count is kept
        const unsigned long long sb = warp_sum_u64(bpart);
        if (lane == 0) sm.red[warp * 4 + 3] = sb;
        __syncthreads();
        if (tid == 0) {
          unsigned long long bb = 0;
          for (int w = 0; w < nwarps; ++w) bb += sm.red[w * 4 + 3];
          PairRaw r;
          r.dis = 0;
          r.ntie = 0;
          r.b = (long long)bb;
          r.g00 = (long long)bb;
          p.raw[slot] = r;
          if (PW) {  // a column without two distinct values: 0 rows -> NA, 1 row -> too short, else single value
            PairComplete c{};
            c.n_rows = (long long)n - XS.n_na - YS.n_na + (long long)bb;
            c.kx = c.ky = 1;
            c.unsupported = absorbed ? 1 : 0;
            p.pw[slot] = c;
          }
        }
        __syncthreads();
        continue;
      }
      // complete-observations mode: the missing rows of x are taken out even if there is only one
      const int f = (PW && XS.n_na > 0) ? XS.n_na : XS.first_run;
      PwSide pwy, pwx;  // y without x's missing rows / x without y's missing rows
      uint32_t ties = 0;
      // Tied x groups other than the first: small ones are compared directly (before anything is
      // written into the sequence buffer), large ones are sorted by y in place after the gather.
      // If the large groups' rank counters would cost more than pass B (very many distinct y
      // values x very many large groups), pass B does all tied rows after pass A instead.
      const int m = XS.n_tied, nlg = XS.flags >> 8;
      const bool by_pass_b = nlg > 0 && p.tier == 2 && (long long)nlg * YS.n_groups > p.budget;
      uint32_t accB = 0;
      // CZ: leave y's rank-0 keys out of pass A only where that takes a whole warp out of its levels (the
      // compacting gather costs more than it saves otherwise).  Compacted, the first ceil(len' / R) ranges are
      // swept, len' = n - (y's rank-0 rows); otherwise all but the floor(lead / R) leading ranges, where the
      // leading block of zero keys is at most the smaller of the two columns' first groups.
      bool cz = false;
      if constexpr (CZ) {
        const int y0 = max(YS.first_run, 1), lead_max = min(XS.first_run, y0);
        cz = ((n - y0 + kkc - 1) / kkc + 31) / 32 < nwarps - lead_max / kkc / 32;
      }
      if constexpr (!RG) {
        if (m > 0 && !by_pass_b)  // keys: 2 m <= 2 cap bytes, the still empty sequence buffer
          small_groups_direct(bufA, m, p.trow + (size_t)xcol * p.nstride, p.tord + (size_t)xcol * p.nstride,
                              rank_tbl, accB, ties);
      }
      // x's first tie group goes in already sorted by y; its joint ties with y fall out of it
      if (!STG && f > 0) {
        if (PW && XS.n_na > 0)
          ties += group_hist<G, true, true, RG>(bufA, cap, f, f, YS.n_groups, permX, rank_tbl, rankY_g, sm.mini,
                                                  sm.fmask, fmask_words(nwarps, kkc) / 3, sm.descT, sm.mini + 16,
                                                  nwarps, p.gstart + (size_t)ycol * p.gstride, YS.n_na, pwy);
        else
          ties += group_hist<G, true, false, RG, CZ>(bufA, cap, f, f, YS.n_groups, permX, rank_tbl, rankY_g, sm.mini,
                                                   sm.fmask, fmask_words(nwarps, kkc) / 3, sm.descT, sm.mini + 16,
                                                   nwarps, nullptr, 0, pwy,
                                                   8 * YS.n_tied <= n,  // y (nearly) tie-free: one bit per rank
                                                   fbXg, sm.nabY, nwords, cz);
      }
      if (PW && YS.n_na > 0)  // the missing rows of y over the ranks of x (read from global memory)
        group_hist<G, false, true, true>(bufA, cap, f, YS.n_na, XS.n_groups, p.perm + (size_t)ycol * p.nstride,
                                         rank_tbl, p.rank + (size_t)xcol * p.nstride, sm.mini, sm.fmask,
                                         fmask_words(nwarps, kkc) / 3, sm.descT, sm.mini + 16, nwarps,
                                         p.gstart + (size_t)xcol * p.gstride, XS.n_na, pwx);
      uint32_t len = (uint32_t)cap, zt = 0u;  // CZ: length of seq', this thread's share of the zero term
      if constexpr (CZ) {
        if (cz)
          len = compact_gather<4>(bufA, rank_tbl, permX, n, f, sm.mini + 18, sm.descT,
                                  reinterpret_cast<uint32_t*>(sm.descB), nwarps, zt);
      }
      if (CZ && cz) {
      } else if (STG) {
        staged_gather(smem_addr(sm.region_ptr), stage_tbl, stage_rows, permX, rankY_g, n, p.nstride, cap, padA, mbar, tma_phase);
      } else {  // seq[q] = rank_y[perm_x[q]] for q >= f, eight positions per thread and step
        auto rk = [&](uint32_t row) -> uint32_t {
          return RG ? (uint32_t)__ldg(rankY_g + row) : M::ld16(M::add(rank_tbl, (int32_t)(row << 1)));
        };
        const uint4* px8 = reinterpret_cast<const uint4*>(permX);
        for (int q8 = (f >> 3) + tid; q8 < (cap >> 3); q8 += T) {
          const int q0 = q8 << 3;
          uint32_t o[4];
          if (q0 + 8 <= n) {
            const uint4 pv = __ldg(px8 + q8);
            const uint32_t pw[4] = {pv.x, pv.y, pv.z, pv.w};
#pragma unroll
            for (int j = 0; j < 4; ++j)
              o[j] = rk(pw[j] & 0xffffu) | (rk(pw[j] >> 16) << 16);
          } else {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const int qa = q0 + 2 * j, qb = qa + 1;
              const uint32_t lo = (qa < n) ? rk(permX[qa]) : padA;
              const uint32_t hi = (qb < n) ? rk(permX[qb]) : padA;
              o[j] = lo | (hi << 16);
            }
          }
          if (q0 >= f) {
            M::st128(M::add(bufA, q0 << 1), o[0], o[1], o[2], o[3]);
          } else {  // the block that straddles f: positions below f belong to the emission
#pragma unroll
            for (int j = 0; j < 8; ++j)
              if (q0 + j >= f) M::st16(M::add(bufA, (q0 + j) << 1), (o[j >> 1] >> ((j & 1) * 16)) & 0xffffu);
          }
        }
      }
      __syncthreads();
      if (RG && m > 0 && !by_pass_b)
        small_groups_inplace<G>(bufA, m, p.tord + (size_t)xcol * p.nstride, p.tpos + (size_t)xcol * p.nstride, accB, ties);
      if ((nlg > 0 || (STG && f > 0)) && !by_pass_b) {
        // large tie groups of x: sorted by y in place (the counters live behind the two pass-A buffers)
        if constexpr (RG)
          ties += large_groups_sorted2<G>(bufA, M::add(bufA, AQ * cap), (p.region_bytes - AQ * cap) >> 2, permX, rankY_g, YS.n_groups,
                                          p.lgrp + (size_t)xcol * kLargeStride, nlg,
                                          reinterpret_cast<uint32_t*>(sm.red), sm.fmask, fmask_words(nwarps, kkc) / 3,
                                          sm.descT, sm.mini + 16, nwarps, STG ? f : 0, sm.mini + 18);
        else
          ties += large_groups_sorted(bufA, M::add(bufA, AQ * cap), (p.region_bytes - AQ * cap) >> 2, permX, rank_tbl, YS.n_groups,
                                      p.lgrp + (size_t)xcol * kLargeStride, nlg,
                                      reinterpret_cast<uint32_t*>(sm.red), sm.fmask, fmask_words(nwarps, kkc) / 3,
                                      sm.descT, sm.mini + 16, nwarps);
      }
      unsigned long long accA = zt;
      // published by the barrier after the gather; a compacted sequence (len' < n <= cap) has no zero keys
      const uint32_t lead = (CZ && len < (uint32_t)cap) ? 0u : sm.mini[18];
      if (IP != 0)
        count_pass_inplace<(IP != 0 ? IP : 1)>(smem_addr(sm.region_ptr), nwarps, L, sm.descT,
                                               reinterpret_cast<uint32_t*>(sm.descB), lane, warp, p.pc, accA, lead);
      else
        count_pass<G, CZ>(bufA, bufB16, kk, nwarps, L, sm.descT, reinterpret_cast<uint32_t*>(sm.descB), lane, warp, p.pc,
                          accA, lead, len, (RX && p.radix) ? sm.region + 4u * (uint32_t)cap : 0u);
      if (IP == 0 && m > 0 && by_pass_b) {
        const int kkB = (((m + 31) >> 5) + nwarps - 1) / nwarps;
        const int capB = (nwarps * kkB) << 5;
        const uint16_t* trow = p.trow + (size_t)xcol * p.nstride;
        const uint16_t* trun = p.trun + (size_t)xcol * p.nstride;
        for (int t = tid; t < capB; t += T)
          M::st32(M::add(bufA, t << 2),
                  (t < m) ? (((uint32_t)trun[t] << 16) | (uint32_t)rankY_g[trow[t]]) : 0xffffffffu);
        __syncthreads();
        bucket_pass<G>(bufA, M::add(bufA, capB << 2), kkB, nwarps, m, L, sm.descT, sm.descB, lane, warp, accB,
                       ties);
      }
      const unsigned long long sA = warp_sum_u64(accA),
                               sB = warp_sum_u64(accB),
                               sT = warp_sum_u64((unsigned long long)ties),
                               sb = warp_sum_u64(((unsigned long long)g00part << 32) | bpart);
      if (lane == 0) {
        sm.red[warp * 4 + 0] = sA;
        sm.red[warp * 4 + 1] = sB;
        sm.red[warp * 4 + 2] = sT;
        sm.red[warp * 4 + 3] = sb;
      }
      __syncthreads();
      long long g_dis = 0, g_ntie = 0, g_b = 0;
      if (tid == 0) {
        unsigned long long a = 0, b2 = 0, t2 = 0, bb = 0;
        for (int w = 0; w < nwarps; ++w) {
          a += sm.red[w * 4 + 0];
          b2 += sm.red[w * 4 + 1];
          t2 += sm.red[w * 4 + 2];
          bb += sm.red[w * 4 + 3];
        }
        PairRaw r;
        r.dis = (long long)(a - YS.cconst - b2);
        r.ntie = (long long)t2;
        r.b = (long long)(bb & 0xffffffffull);
        r.g00 = absorbed ? (long long)(bb >> 32) : r.b;
        p.raw[slot] = r;
        g_dis = r.dis;
        g_ntie = r.ntie;
        g_b = r.b;
      }
      if (PW) {
        unsigned long long kxy = ((unsigned long long)pwx.k << 32) | pwy.k, z0 = 0, z1 = 0;
        block_sum4(sm.red, nwarps, pwy.S, pwy.T, pwx.S, pwx.T);
        block_sum4(sm.red, nwarps, pwy.s2, pwy.s3, pwy.s5, kxy);
        block_sum4(sm.red, nwarps, pwx.s2, pwx.s3, pwx.s5, z0);
        (void)z1;
        if (tid == 0) {
          const long long ax = XS.n_na, ay = YS.n_na, b = g_b;
          const long long xm = ax - b, ym = ay - b;  // missing in x only / in y only
          const long long t1 = ax > 0 ? (long long)pwy.T : 0, t2 = ay > 0 ? (long long)pwx.T : 0;
          // discordant pairs of the global count with a row missing in one column (NA below every
          // value): x-missing row above a shared row in y, shared row below a y-missing row in x,
          // x-missing row against y-missing row
          const long long c1 = ax > 0 ? (long long)pwy.S - xm * (xm - 1) / 2 + t1 : 0;
          const long long c2 = ay > 0 ? (long long)pwx.S - ym * (ym - 1) / 2 + t2 : 0;
          PairComplete c{};
          c.n_rows = (long long)n - ax - ay + b;
          c.dis = g_dis - c1 - c2 - xm * ym;
          c.ntie = g_ntie - b * (b - 1) / 2 - t1 - t2;
          if (ay > 0) {
            c.xs2 = (long long)pwx.s2; c.xs3 = (long long)pwx.s3; c.xs5 = (long long)pwx.s5;
            c.kx = (int32_t)(kxy >> 32);
          } else {
            c.xs2 = XS.s2o; c.xs3 = XS.s3o; c.xs5 = XS.s5o;
            c.kx = XS.n_groups - (ax > 0 ? 1 : 0);
          }
          if (ax > 0) {
            c.ys2 = (long long)pwy.s2; c.ys3 = (long long)pwy.s3; c.ys5 = (long long)pwy.s5;
            c.ky = (int32_t)(kxy & 0xffffffffull);
          } else {
            c.ys2 = YS.s2o; c.ys3 = YS.s3o; c.ys5 = YS.s5o;
            c.ky = YS.n_groups - (ay > 0 ? 1 : 0);
          }
          c.unsupported = absorbed ? 1 : 0;
          p.pw[slot] = c;
        }
      }
      __syncthreads();
    }
    __syncthreads();  // unit_slot is rewritten at the top of the loop
  }
}

// cconst of every column: the raw pass-A count of the column's own sorted rank sequence
// (no inversions), evaluated by the same code path as the pair kernel.  Grid-stride over columns.
template <bool G>
__global__ void __launch_bounds__(1024, 1) column_const_kernel(const TiledParams p, ColStats* stats, int c0, int C) {
  typedef Mem<G> M;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int T = blockDim.x, nwarps = T >> 5;
  const int n = p.n, kk = p.kk;
  const int cap = (nwarps * kk) << 8;
  Carve sm(smem_raw, p.wstride, fmask_words(nwarps, kk << 3));
  const typename M::ptr bufA = region_base<G>(sm, p), bufB = M::add(bufA, 2 * cap);
  for (int col = c0 + blockIdx.x; col < C; col += gridDim.x) {
    const ColStats CS = stats[col];
    if (CS.n_groups < 2) {
      if (tid == 0) stats[col].cconst = 0;
      continue;
    }
    const uint16_t* pm = p.perm + (size_t)col * p.nstride;
    const uint16_t* rk = p.rank + (size_t)col * p.nstride;
    const uint32_t padA = (1u << CS.levels) - 1u;
    for (int q = tid; q < cap; q += T) M::st16(M::add(bufA, q << 1), (q < n) ? (uint32_t)rk[pm[q]] : padA);
    __syncthreads();
    unsigned long long accA = 0;
    count_pass<G>(bufA, bufB, kk, nwarps, CS.levels, sm.descT, reinterpret_cast<uint32_t*>(sm.descB), lane, warp, p.pc, accA,
                  0u, 0u, (!G && p.radix) ? sm.region + 4u * (uint32_t)cap : 0u);
    const unsigned long long s = warp_sum_u64(accA);
    if (lane == 0) sm.red[warp] = s;
    __syncthreads();
    if (tid == 0) {
      unsigned long long a = 0;
      for (int w = 0; w < nwarps; ++w) a += sm.red[w];
      stats[col].cconst = a;
    }
    __syncthreads();
  }
}

// ---- K2-naive: one thread per pair, the reference's Fenwick algorithm ---------------------
// (src/kendallc.cpp:70-100) on the precomputed ranks, Fenwick array and a per-group counter
// array in global memory.  This is the internal baseline BASELINE.json names and an
// independent on-device cross-check of the tiled kernel.
__global__ void pairs_naive_kernel(const TiledParams p, long long P, uint32_t* scratch,
                                   long long n_threads) {
  const long long tid0 = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (tid0 >= n_threads) return;
  const int n = p.n;
  uint32_t* bit = scratch + (size_t)tid0 * (2 * (size_t)n + 2);  // Fenwick tree, 1-based
  uint32_t* cnt = bit + n + 1;                                    // joint-tie counters per y rank
  // thread t takes units t, t + n_threads, ...
  for (long long u = tid0; u < p.n_units; u += n_threads) {
    const PairUnit unit = p.units[u];
    for (int k = 0; k < unit.count; ++k) {
      const long long slot = unit.slot0 + k;
      const int ycol = unit.col;
      const int xcol = unit.j_explicit ? p.pj_list[slot] : unit.j0 + k;
      const ColStats XS = p.stats[xcol], YS = p.stats[ycol];
      PairRaw r;
      r.dis = 0;
      r.ntie = 0;
      r.b = 0;
      r.g00 = 0;
      if (XS.n_groups >= 2 && YS.n_groups >= 2) {
        const uint16_t* permX = p.perm + (size_t)xcol * p.nstride;
        const uint16_t* rankX = p.rank + (size_t)xcol * p.nstride;
        const uint16_t* rankY = p.rank + (size_t)ycol * p.nstride;
        const int sup = YS.n_groups + 1;
        for (int i = 0; i <= sup; ++i) bit[i] = 0;
        for (int i = 0; i < sup; ++i) cnt[i] = 0;
        long long dis = 0, ntie = 0;
        int i = 0, kk = 0;
        while (i < n) {
          const int xg = rankX[permX[i]];
          while (kk < n && rankX[permX[kk]] == xg) {  // query the whole x group first
            dis += i;
            int idx = (int)rankY[permX[kk]] + 1;
            ntie += cnt[idx - 1]++;
            while (idx != 0) {
              dis -= bit[idx];
              idx &= idx - 1;
            }
            ++kk;
          }
          while (i < kk) {  // then insert it
            int idx = (int)rankY[permX[i]] + 1;
            cnt[idx - 1] = 0;
            while (idx < sup) {
              bit[idx] += 1;
              idx += idx & (-idx);
            }
            ++i;
          }
        }
        r.dis = dis;
        r.ntie = ntie;
      }
      {
        const uint32_t* nbX = p.nabits + (size_t)xcol * p.wstride;
        const uint32_t* nbY = p.nabits + (size_t)ycol * p.wstride;
        const uint32_t* g0X = ((XS.flags & 1) ? p.firstbits : p.nabits) + (size_t)xcol * p.wstride;
        const uint32_t* g0Y = ((YS.flags & 1) ? p.firstbits : p.nabits) + (size_t)ycol * p.wstride;
        long long b = 0, g00 = 0;
        for (int w = 0; w < (p.n32 >> 5); ++w) {
          b += __popc(nbX[w] & nbY[w]);
          g00 += __popc(g0X[w] & g0Y[w]);
        }
        r.b = b;
        r.g00 = g00;
      }
      p.raw[slot] = r;
    }
  }
}

// ---- K3: fp64 epilogue -------------------------------------------------------------------
struct EpiParams {
  const ColStats* stats;
  const PairUnit* units;
  const int32_t* pj_list;
  const PairRaw* raw;
  const PairComplete* pw;  // complete-observations mode (else null)
  double* tau;
  double* pvalue;
  double* taumax;
  double* completeness;
  int32_t* status;
  long long* counts;
  unsigned long long* max_bits;
  long long n_units;
  long long n;
  int perspective, alternative, continuity;
  int lane_shift;  // 2^lane_shift threads per unit (the smallest power of two that covers the longest unit)
};

__global__ void __launch_bounds__(128) epilogue_kernel(const EpiParams p) {
  // 2^lane_shift consecutive threads per unit, one pair per thread and step
  const long long gt = (long long)blockIdx.x * 128 + threadIdx.x;
  const long long u = gt >> p.lane_shift;
  const int lane = threadIdx.x & 31, sub = (int)(gt & ((1 << p.lane_shift) - 1));
  double mx = -1.0;
  if (u < p.n_units) {
    const PairUnit unit = p.units[u];
    for (int k = sub; k < unit.count; k += 1 << p.lane_shift) {
      const long long slot = unit.slot0 + k;
      const int xcol = unit.j_explicit ? p.pj_list[slot] : unit.j0 + k;
      PairRaw r = p.raw[slot];
      PairOut o;
      if (p.pw) {
        // the kernel's x is the second column of the pair; the reference names the first one x
        PairComplete c = p.pw[slot], d = c;
        d.xs2 = c.ys2; d.xs3 = c.ys3; d.xs5 = c.ys5; d.kx = c.ky;
        d.ys2 = c.xs2; d.ys3 = c.xs3; d.ys5 = c.xs5; d.ky = c.kx;
        pair_epilogue_complete(d, p.alternative, p.continuity, o);
        r.dis = c.dis;
        r.b = 0;
      } else {
        // reference naming: x = first column of the pair (unit.col), y = the second
        pair_epilogue(p.n, p.stats[unit.col], p.stats[xcol], r.dis, r.ntie, r.b, r.g00, p.perspective,
                      p.alternative, p.continuity, o);
      }
      p.tau[slot] = o.tau;
      if (p.pvalue) p.pvalue[slot] = o.pvalue;
      if (p.taumax) p.taumax[slot] = o.taumax;
      if (p.completeness) p.completeness[slot] = o.completeness;
      if (p.status) p.status[slot] = o.status;
      if (p.counts) {
        long long* c = p.counts + 7 * slot;
        c[0] = r.dis;
        c[1] = o.ntie;
        c[2] = o.xtie;
        c[3] = o.ytie;
        c[4] = o.tot;
        c[5] = o.n_entry;
        c[6] = r.b;
      }
      if (o.status == 0 && o.taumax == o.taumax) mx = fmax(mx, o.taumax);
    }
  }
#pragma unroll
  for (int d = 16; d >= 1; d >>= 1) mx = fmax(mx, __shfl_xor_sync(FULL, mx, d));
  // tau_max >= 0, so the IEEE bit pattern orders like an unsigned integer
  if (lane == 0 && mx >= 0.0) atomicMax(p.max_bits, (unsigned long long)__double_as_longlong(mx));
}

__global__ void pnorm_kernel(const double* z, long long n, int lower, double* out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = pnorm_std(z[i], lower != 0);
}


// ---- shared-memory bandwidth microbenchmark (roofline denominator) -----------------------
// Conflict-free sweep: every thread loads one word (or one uint4) and stores one per step.
template <typename T>
__global__ void __launch_bounds__(1024) smem_sweep_kernel(int iters, unsigned* sink) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  T* s = reinterpret_cast<T*>(smem_raw);
  constexpr int N = 4096;  // elements of T per CTA
  const int tid = threadIdx.x;
  for (int i = tid; i < N; i += 1024) s[i] = T{};
  __syncthreads();
  T a0 = s[tid], a1 = s[tid + 1024], a2 = s[tid + 2048], a3 = s[tid + 3072];
  for (int it = 0; it < iters; ++it) {
    s[tid] = a1;
    s[tid + 1024] = a2;
    s[tid + 2048] = a3;
    s[tid + 3072] = a0;
    __syncwarp();
    a0 = s[tid];
    a1 = s[tid + 1024];
    a2 = s[tid + 2048];
    a3 = s[tid + 3072];
    __syncwarp();
  }
  s[tid] = a0;
  s[tid + 1024] = a1;
  s[tid + 2048] = a2;
  s[tid + 3072] = a3;
  __syncthreads();
  if (tid == 0) sink[blockIdx.x] = *reinterpret_cast<unsigned*>(&s[blockIdx.x & 1023]);
}

template <typename T>
double run_smem_sweep(int n_sm, unsigned* d_sink) {
  const int iters = 4000;
  const size_t smem = sizeof(T) * 4096;
  auto kern = smem_sweep_kernel<T>;
  if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return -1;
  const int grid = n_sm * 2;
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0);
  cudaEventCreate(&e1);
  kern<<<grid, 1024, smem>>>(iters / 10, d_sink);  // warm-up
  double best = 0;
  for (int rep = 0; rep < 5; ++rep) {
    cudaEventRecord(e0);
    kern<<<grid, 1024, smem>>>(iters, d_sink);
    cudaEventRecord(e1);
    if (cudaEventSynchronize(e1) != cudaSuccess) { best = -1; break; }
    float ms = 0;
    cudaEventElapsedTime(&ms, e0, e1);
    const double bytes = (double)grid * 1024.0 * iters * 4.0 * 2.0 * sizeof(T);  // 4 loads + 4 stores
    best = std::max(best, bytes / (ms * 1e-3) / 1e9);
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  return best;
}

// ---- instruction-issue microbenchmark (the second roofline denominator) ---------------------
// The pair kernel is bound by instruction issue on the two integer-capable pipes: the ALU pipe
// (LOP3 / IADD3 / SHF / SEL / PRMT) and the FMA pipe (IMAD), each taking one warp instruction every
// other cycle per scheduler.  MODE 0: LOP3 only, 1: IMAD only, 2: the two interleaved.  Eight
// independent chains per thread hide the 4-cycle latency; 32 warps per SM keep every scheduler fed.
template <int MODE>
__global__ void __launch_bounds__(1024) issue_sweep_kernel(int iters, uint32_t m, uint32_t* sink) {
  uint32_t a[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) a[k] = threadIdx.x * 2654435761u + (uint32_t)k * 40503u + blockIdx.x;
  uint32_t b = m | 1u, c = m ^ 0x9e3779b9u;
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int rep = 0; rep < 8; ++rep) {
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const bool fma = MODE == 1 || (MODE == 2 && (k & 1));
        if (fma)
          asm volatile("mad.lo.u32 %0, %0, %1, %2;" : "+r"(a[k]) : "r"(b), "r"(c));
        else
          asm volatile("lop3.b32 %0, %0, %1, %2, 0x96;" : "+r"(a[k]) : "r"(b), "r"(c));
      }
    }
  }
  uint32_t x = 0;
#pragma unroll
  for (int k = 0; k < 8; ++k) x ^= a[k];
  if (x == 0x12345u) sink[0] = x;  // keeps the chains alive
}

template <int MODE>
double run_issue_sweep(int n_sm, uint32_t* d_sink) {
  const int iters = 4000, grid = n_sm * 2;
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0);
  cudaEventCreate(&e1);
  issue_sweep_kernel<MODE><<<grid, 1024>>>(iters / 10, 3u, d_sink);
  double best = 0;
  for (int rep = 0; rep < 5; ++rep) {
    cudaEventRecord(e0);
    issue_sweep_kernel<MODE><<<grid, 1024>>>(iters, 3u, d_sink);
    cudaEventRecord(e1);
    if (cudaEventSynchronize(e1) != cudaSuccess) { best = -1; break; }
    float ms = 0;
    cudaEventElapsedTime(&ms, e0, e1);
    const double warp_inst = (double)grid * 32.0 * iters * 64.0;  // 64 instructions per thread and iteration
    best = std::max(best, warp_inst / (ms * 1e-3) / 1e9);
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  return best;
}

TiledParams make_params(const PairLaunch& pl) {
  const ColumnTables& t = *pl.tab;
  TiledParams p;
  p.perm = t.perm;
  p.rank = t.rank;
  p.trow = t.trow;
  p.trun = t.trun;
  p.tord = t.tord;
  p.tpos = t.tend;
  p.nabits = t.nabits;
  p.firstbits = t.firstbits;
  p.stats = t.stats;
  p.units = pl.units;
  p.pj_list = pl.pj_list;
  p.raw = pl.raw;
  p.pw = pl.pw;
  p.gstart = t.gstart;
  p.gstride = (int)t.gstride;
  p.lgrp = t.lgrp;
  p.region_bytes = 0;
  p.unit_counter = pl.unit_counter;
  p.n_units = pl.n_units;
  p.n = (int)t.n;
  p.n32 = (int)((t.n + 31) & ~31LL);
  p.nstride = (int)t.nstride;
  p.wstride = (int)t.wstride;
  p.scratch = nullptr;
  p.scratch_stride = 0;
  p.kk = 0;
  p.radix = false;
  p.max_tied = t.max_tied;
  p.tier = 0;
  p.budget = 16LL * t.n;
  p.pc = make_pipe_const();
  return p;
}

}  // namespace

int64_t tiled_max_n() { return 65535; }

int measure_smem_bandwidth(double* gbps32, double* gbps128) {
  int dev = 0, n_sm = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return -1;
  if (cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return -1;
  unsigned* d_sink = nullptr;
  if (cudaMalloc(reinterpret_cast<void**>(&d_sink), sizeof(unsigned) * n_sm * 2) != cudaSuccess) return -1;
  const double a = run_smem_sweep<unsigned>(n_sm, d_sink);
  const double b = run_smem_sweep<uint4>(n_sm, d_sink);
  cudaFree(d_sink);
  if (a < 0 || b < 0) return -1;
  *gbps32 = a;
  *gbps128 = b;
  return 0;
}

int measure_issue_rate(double* alu, double* fma, double* mixed) {
  int dev = 0, n_sm = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return -1;
  if (cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return -1;
  uint32_t* d_sink = nullptr;
  if (cudaMalloc(reinterpret_cast<void**>(&d_sink), sizeof(uint32_t) * 4) != cudaSuccess) return -1;
  const double a = run_issue_sweep<0>(n_sm, d_sink), f = run_issue_sweep<1>(n_sm, d_sink),
               m = run_issue_sweep<2>(n_sm, d_sink);
  cudaFree(d_sink);
  if (a < 0 || f < 0 || m < 0) return -1;
  *alu = a;
  *fma = f;
  *mixed = m;
  return 0;
}

// Pass A's low-nibble level counts a thread's 8 kk keys in byte fields (NibbleCounts): 8 kk <= 255
constexpr int kMaxRuns = 31;

// 8-key runs per thread such that W warps cover n keys: the smallest odd count (bank-conflict-free
// 128-bit loads), unless that pushes the padded length past the 65536 slots the packed 16-bit
// slot indices of pass A can address; then the smallest count, or 0 if W cannot cover n at all.
static int odd_runs(int64_t n, int W) {
  int kk = (int)((n + 256LL * W - 1) / (256LL * W));
  if (kk < 1) kk = 1;
  if (256LL * W * (kk | 1) <= 65536) return kk | 1;
  return 256LL * W * kk <= 65536 ? kk : 0;
}

// warps per CTA of the per-column constant kernel: 16..32, least padding (the constant does not
// depend on the launch shape)
static int const_warps(int64_t n) {
  int W = 32;
  long long best = -1;
  for (int w = 32; w >= 16; --w) {
    const long long cap = 256LL * w * odd_runs(n, w);
    if (cap > 0 && (best < 0 || cap < best)) { best = cap; W = w; }
  }
  return W;
}

// Pass A's radix-16 levels (count_pass, radix_level) need, behind the two sequence buffers, a u16 slot counter per
// digit and thread (plus the 64 bytes its odd threads' last row runs over) and 32 bytes of node totals per warp
static int radix_area_bytes(int W) { return 16 * 2 * 32 * W + 64 + 32 * W; }
// region of the per-column constant kernel: its two sequence buffers and, with radix levels, their counter area
static int const_region(int64_t n, int W, bool radix) {
  return (2 * 2 * (W * odd_runs(n, W) * 256) + (radix ? radix_area_bytes(W) : 0) + 15) & ~15;
}

// Launch shape for vectors of length n: warps per CTA, 8-key runs per thread (odd), bytes of the
// ping-pong region (pass A: two u16 buffers; pass B: two u32 buffers sized for the largest tied
// list), and whether the region fits shared memory or has to live in the global scratch.
// `radix`: pass A runs radix-16 levels, the region holds their counter area behind the two buffers.
static TiledShape shape_for(int64_t n, int tier, int64_t wstride, int n_sm, int64_t n_units, bool allow_inplace,
                            bool radix) {
  TiledShape sh;
  sh.radix = radix;
  // pass A: two u16 buffers (4*cap bytes).  Tier 1 adds a quarter more (cap bytes) for the rank
  // counters of the large tie groups -- a larger counter area means fewer rounds over the large
  // groups but fewer CTAs per SM, which measured worse (profiles/).  Tier 2: twice as much for
  // pass B's two u32 buffers.  The radix levels' counters use what lies behind the two buffers
  // (free during pass A) and extend the region where that is too small.
  auto quarters_of = [&](int) { return tier == 0 ? 4 : tier == 1 ? 5 : 8; };
  auto region_of = [&](int w) {
    const int cap = w * odd_runs(n, w) * 256;
    return (std::max(quarters_of(w) * cap, radix ? 4 * cap + radix_area_bytes(w) : 0) + 15) & ~15;
  };
  auto smem_of = [&](int w) {
    return tiled_smem_bytes(region_of(w), (int)wstride, fmask_words(w, odd_runs(n, w) << 3));
  };
  // W: padded length (odd run count) x per-level fixed cost (two barriers and two scans cost
  // about two runs per thread) x a latency-hiding factor for fewer than 32 resident warps per
  // SM.  Fitted to the B200 sweeps in profiles/.  Shapes that do not fit shared memory run 32
  // warps on the global scratch.
  int W = 32;
  double best = 1e300;
  for (int w = 1; w <= 32; ++w) {
    const int kk = odd_runs(n, w);
    if (kk == 0 || kk > kMaxRuns) continue;
    const size_t smem = smem_of(w);
    if (smem > 227 * 1024) continue;
    // resident CTAs per SM: threads, shared memory, registers (64 per thread in the roomy class)
    const int ctas = std::max(1, (int)std::min<size_t>(std::min(std::min(32, 2048 / (32 * w)), 32 / w),
                                                       (228 * 1024) / (smem + 1024)));
    const double rw = std::min(32.0, (double)w * ctas);
    double cost = 256.0 * w * kk * (1.0 + 2.0 / kk) * std::pow(32.0 / rw, 0.4);
    if (n_units > 0) {  // small jobs: whole rounds of equal-cost pairs over the resident CTAs
      const double per_cta = (double)n_units / ((double)n_sm * ctas);
      if (per_cta < 64.0) cost *= std::ceil(per_cta) / per_cta;
    }
    if (cost < best) { best = cost; W = w; }
  }
  if (const char* e = getenv("ICIKT_WARPS")) {
    const int v = atoi(e);
    if (v >= 1 && v <= 32 && odd_runs(n, v) > 0 && odd_runs(n, v) <= kMaxRuns) W = v;
  }
  if (getenv("ICIKT_FORCE_GMEM")) W = 32;
  sh.warps = W;
  sh.kk = odd_runs(n, W);
  sh.region_bytes = region_of(W);
  if (best >= 1e300 && tier <= 1 && allow_inplace && !getenv("ICIKT_FORCE_GMEM") && !getenv("ICIKT_WARPS")) {
    // nothing fits shared memory with two sequence buffers: the in-place variant (one buffer,
    // the keys of a level held in registers, kk fixed at compile time) takes up to 28 warps
    constexpr int KK = 9;
    const int w = (int)((n + 256LL * KK - 1) / (256LL * KK));
    const int cap = 256 * KK * std::max(w, 1);
    const int region = ((tier == 0 ? 2 : 3) * cap + 15) & ~15;
    if (w >= 1 && w <= 28 && cap <= 65536 &&
        tiled_smem_bytes(region, (int)wstride, fmask_words(w, KK << 3)) <= 227 * 1024) {
      sh.inplace_kk = KK;
      sh.warps = W = w;
      sh.kk = KK;
      sh.region_bytes = region;
      {
        // one CTA per SM either way: the rank counters of the tie groups take all that is left (more groups
        // per round); before that the area stages y's rank table for the gather (tier 0 as well: the first
        // group is sorted there)
        const size_t fixed = tiled_smem_bytes(0, (int)wstride, fmask_words(w, KK << 3));
        sh.region_bytes = (int)((227 * 1024 - fixed) & ~size_t(15));
      }
    }
  }
  {  // the per-column constant kernel has its own shape: its pass-A buffers must fit a scratch slot too
    const int Wc = const_warps(n);
    sh.const_region_bytes = const_region(n, Wc, radix);
    sh.const_gmem = tiled_smem_bytes(sh.const_region_bytes, (int)wstride, fmask_words(Wc, odd_runs(n, Wc) << 3)) > 227 * 1024 ||
                    getenv("ICIKT_FORCE_GMEM") != nullptr;
  }
  sh.gmem = sh.inplace_kk == 0 && (smem_of(W) > 227 * 1024 || getenv("ICIKT_FORCE_GMEM") != nullptr);
  sh.max_ctas = n_sm * std::max(1, 2048 / (32 * W));
  return sh;
}

// Pass A's level structure is part of every column's constant cconst, so it follows from n alone, the same
// for all three tiers and the constant kernel: radix-16 levels where each of them runs the two-buffer kernel
// in shared memory with the counter area, above the lengths the fused column kernel covers (its pass keeps
// the two-bit levels).  The tuning knobs that pin a shape (ICIKT_WARPS, ICIKT_FORCE_GMEM) act in shape_for, so
// a pinned shape that leaves shared memory keeps the two-bit levels for every tier.
static bool pass_a_radix(int64_t n, int64_t wstride) {
  if (n <= 8192) return false;
  for (int tier = 0; tier <= 2; ++tier) {
    const TiledShape sh = shape_for(n, tier, wstride, 1, 0, true, true);
    if (sh.gmem || sh.inplace_kk != 0 || sh.const_gmem) return false;
  }
  return true;
}

TiledShape tiled_shape(int64_t n, int tier, int64_t wstride, int n_sm, int64_t n_units, bool allow_inplace) {
  return shape_for(n, tier, wstride, n_sm, n_units, allow_inplace, pass_a_radix(n, wstride));
}

namespace {

template <int MAXT, int MINB, bool G, bool PW = false, int IP = 0, bool CZ = false>
int tiled_occupancy(int threads, size_t smem) {
  auto kern = pairs_tiled_kernel<MAXT, MINB, G, PW, IP, CZ>;
  if (threads > MAXT) return 0;
  // always the architectural maximum, never the shape's own need: the attribute is per device, and two
  // host threads driving plans of different shapes on one device must not shrink it under each other
  // between the query and the launch
  (void)smem;
  if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024) != cudaSuccess) {
    g_launch_error = cudaGetLastError();
    g_launch_note = "cudaFuncSetAttribute(max dynamic shared memory)";
    return 0;
  }
  int per_sm = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, threads, smem) != cudaSuccess) {
    g_launch_error = cudaGetLastError();
    g_launch_note = "cudaOccupancyMaxActiveBlocksPerMultiprocessor";
    return 0;
  }
  return per_sm;
}

template <int MAXT, int MINB, bool G, bool PW = false, int IP = 0, bool CZ = false>
int launch_tiled_variant(const TiledParams& p, int threads, long long grid, size_t smem, cudaStream_t stream) {
  pairs_tiled_kernel<MAXT, MINB, G, PW, IP, CZ><<<(unsigned)grid, threads, smem, stream>>>(p);
  return launch_status(1);
}

// Three register classes of the same code (64 / 40 / 32 registers per thread): take the roomiest
// one unless a tighter class keeps clearly more threads resident for this shared-memory footprint.
template <bool G, bool CZ>
int launch_tiled_cls(const TiledParams& p, const TiledShape& sh, size_t smem, int n_sm, cudaStream_t stream);

template <bool G>
int launch_tiled_g(TiledParams& p, const TiledShape& sh, size_t smem, int n_sm, cudaStream_t stream) {
  const int threads = 32 * sh.warps;
  if (!G && sh.inplace_kk == 9) {  // long vectors in place: 28 warps at most, ~72 registers
    const int occ = tiled_occupancy<896, 1, false, false, 9>(threads, smem);
    if (occ < 1) return launch_refused("the in-place pair kernel does not fit an SM (occupancy 0)");
    long long grid = std::max<long long>(1, std::min<long long>((long long)n_sm * occ, p.n_units));
    return launch_tiled_variant<896, 1, false, false, 9>(p, threads, grid, smem, stream);
  }
  if (p.pw) {  // complete-observations mode: one register class
    const int occ = tiled_occupancy<1024, 1, G, true>(threads, smem);
    if (occ < 1) return launch_refused("the complete-observations pair kernel does not fit an SM (occupancy 0)");
    long long grid = (long long)n_sm * occ;
    if (grid > p.n_units) grid = p.n_units;
    if (G && grid > sh.scratch_ctas) grid = sh.scratch_ctas;
    if (grid < 1) grid = 1;
    return launch_tiled_variant<1024, 1, G, true>(p, threads, grid, smem, stream);
  }
  // tier 0 in shared memory with 8 or more warps may run pass A on the sequence without y's lowest-rank keys
  // (decided per pair).  Below that the compacting instantiation measured slower on a B200 although it compacts
  // nothing there (1-4 warps at n = 2 000 ... 6 887: 0.4-1.7 %); at 16 warps (n = 20 000) it gains 4.7 %.
  if (!G && p.tier == 0 && sh.warps >= 8) return launch_tiled_cls<G, !G>(p, sh, smem, n_sm, stream);
  return launch_tiled_cls<G, false>(p, sh, smem, n_sm, stream);
}

template <bool G, bool CZ>
int launch_tiled_cls(const TiledParams& p, const TiledShape& sh, size_t smem, int n_sm, cudaStream_t stream) {
  const int threads = 32 * sh.warps;
  const int o64 = tiled_occupancy<1024, 1, G, false, 0, CZ>(threads, smem);
  const int o40 = tiled_occupancy<512, 3, G, false, 0, CZ>(threads, smem);
  const int o32 = tiled_occupancy<1024, 2, G, false, 0, CZ>(threads, smem);
  // the tighter classes spill: they have to buy at least a quarter more resident CTAs
  int cls = 0, best = o64;
  if (!p.radix && 4 * o40 >= 5 * best) { cls = 1; best = o40; }
  if (!p.radix && 4 * o32 >= 5 * best) { cls = 2; best = o32; }
  if (const char* e = getenv("ICIKT_REGCLASS"); e && !p.radix) {
    const int v = atoi(e);
    if (v == 0 && o64 > 0) { cls = 0; best = o64; }
    if (v == 1 && o40 > 0) { cls = 1; best = o40; }
    if (v == 2 && o32 > 0) { cls = 2; best = o32; }
  }
  if (best < 1) {
    if (g_launch_error != cudaSuccess) return -1;  // the occupancy query itself failed: keep its error
    return launch_refused("the pair kernel does not fit an SM (occupancy 0 in every register class)");
  }
  long long grid = (long long)n_sm * best;
  if (grid > p.n_units) grid = p.n_units;
  if (G && grid > sh.scratch_ctas) grid = sh.scratch_ctas;
  if (grid < 1) grid = 1;
  if (cls == 2) return launch_tiled_variant<1024, 2, G, false, 0, CZ>(p, threads, grid, smem, stream);
  if (cls == 1) return launch_tiled_variant<512, 3, G, false, 0, CZ>(p, threads, grid, smem, stream);
  return launch_tiled_variant<1024, 1, G, false, 0, CZ>(p, threads, grid, smem, stream);
}

}  // namespace

int launch_pairs_tiled(const PairLaunch& pl, const TiledShape& sh, int n_sm, int tier, cudaStream_t stream) {
  TiledParams p = make_params(pl);
  p.tier = tier;
  p.kk = sh.kk;
  p.region_bytes = sh.region_bytes;
  p.radix = sh.radix;
  p.scratch = pl.scratch;
  p.scratch_stride = sh.scratch_stride;
  const int fw = fmask_words(sh.warps, sh.kk << 3);
  if (sh.gmem) {
    if (!pl.scratch || sh.region_bytes > sh.scratch_stride) return -2;
    return launch_tiled_g<true>(p, sh, tiled_smem_bytes(0, p.wstride, fw), n_sm, stream);
  }
  return launch_tiled_g<false>(p, sh, tiled_smem_bytes(sh.region_bytes, p.wstride, fw), n_sm, stream);
}

int launch_column_consts(ColumnTables& tab, const TiledShape& sh, unsigned char* scratch, cudaStream_t stream,
                         int64_t col_lo, int64_t col_hi) {
  PairLaunch pl{};
  pl.tab = &tab;
  TiledParams p = make_params(pl);
  const int W = const_warps(tab.n);
  p.kk = odd_runs(tab.n, W);
  p.radix = sh.radix;
  const int region = const_region(tab.n, W, sh.radix);
  const int fw = fmask_words(W, p.kk << 3);
  const bool g = tiled_smem_bytes(region, p.wstride, fw) > 227 * 1024 || getenv("ICIKT_FORCE_GMEM") != nullptr;
  long long grid = col_hi - col_lo;
  if (grid <= 0) return 0;
  if (g) {
    if (!scratch || sh.scratch_stride < region) return -2;  // the plan sizes the slot as max(region, const region)
    p.scratch = scratch;
    p.scratch_stride = sh.scratch_stride;
    grid = std::min<long long>(grid, sh.scratch_ctas);
    const size_t smem = tiled_smem_bytes(0, p.wstride, fw);
    if (cudaFuncSetAttribute(column_const_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024) != cudaSuccess) return -1;
    column_const_kernel<true><<<(unsigned)grid, 32 * W, smem, stream>>>(p, tab.stats, (int)col_lo, (int)col_hi);
  } else {
    const size_t smem = tiled_smem_bytes(region, p.wstride, fw);
    if (cudaFuncSetAttribute(column_const_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024) != cudaSuccess) return -1;
    column_const_kernel<false><<<(unsigned)grid, 32 * W, smem, stream>>>(p, tab.stats, (int)col_lo, (int)col_hi);
  }
  return launch_status(1);
}

size_t naive_scratch_bytes(int64_t n, int64_t n_threads) {
  return sizeof(uint32_t) * (size_t)n_threads * (2 * (size_t)n + 2);
}

int launch_pairs_naive(const PairLaunch& pl, int64_t P, uint32_t* d_scratch, int64_t n_threads,
                       cudaStream_t stream) {
  const TiledParams p = make_params(pl);
  const int block = 128;
  const long long grid = (n_threads + block - 1) / block;
  pairs_naive_kernel<<<(unsigned)grid, block, 0, stream>>>(p, P, d_scratch, n_threads);
  return launch_status(1);
}

int launch_epilogue(const EpilogueLaunch& el, cudaStream_t stream) {
  EpiParams p;
  p.stats = el.tab->stats;
  p.units = el.units;
  p.pj_list = el.pj_list;
  p.raw = el.raw;
  p.pw = el.pw;
  p.tau = el.tau;
  p.pvalue = el.pvalue;
  p.taumax = el.taumax;
  p.completeness = el.completeness;
  p.status = el.status;
  p.counts = reinterpret_cast<long long*>(el.counts);
  p.max_bits = el.max_taumax_bits;
  p.n_units = el.n_units;
  p.n = el.tab->n;
  p.perspective = el.perspective;
  p.alternative = el.alternative;
  p.continuity = el.continuity;
  if (el.n_units <= 0) return 0;
  p.lane_shift = 0;
  while ((1 << p.lane_shift) < el.max_unit_pairs && p.lane_shift < 5) ++p.lane_shift;
  const long long grid = ((el.n_units << p.lane_shift) + 127) / 128;
  epilogue_kernel<<<(unsigned)grid, 128, 0, stream>>>(p);
  return launch_status(1);
}

int launch_pnorm(const double* d_z, int64_t n, int lower, double* d_out, cudaStream_t stream) {
  if (n <= 0) return 0;
  pnorm_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(d_z, n, lower, d_out);
  return launch_status(1);
}

}  // namespace icikt
