// icikt_reshape.cu -- the result formats either side of the pair kernel, on the device:
//   * scale_and_reshape (R/kendalltau.R:357-421): per-pair results -> symmetric C x C matrices,
//     cor = raw / max(taumax), the diagonal of diag_good (:374-386);
//   * pairwise_completeness (R/kendalltau.R:563-629): missing-row bit masks and popc(x | y);
//   * CSC (sparse) input expanded into the dense column-major matrix the column kernels read.
// All of it is HBM-bound byte moving; nothing here touches shared memory or tensor cores.
#include "icikt_internal.h"

namespace icikt {

namespace {

constexpr unsigned FULL = 0xffffffffu;

struct FillParams {
  MatrixFill f;
  int lane_shift;
};

// Same thread-to-pair mapping as the epilogue kernel: 2^lane_shift consecutive threads per unit,
// so the writes m[j + i*C] of one unit (consecutive j) coalesce; the mirrored writes m[i + j*C]
// are one 8-byte store per column.
__global__ void __launch_bounds__(128) matrix_fill_kernel(const FillParams p) {
  const MatrixFill& f = p.f;
  const long long gt = (long long)blockIdx.x * 128 + threadIdx.x;
  const long long u = gt >> p.lane_shift;
  const int sub = (int)(gt & ((1 << p.lane_shift) - 1));
  if (u >= f.n_units) return;
  const PairUnit unit = f.units[u];
  const unsigned long long bits = *f.max_taumax_bits;
  // max(taumax, na.rm = TRUE) of the computed pairs (R/kendalltau.R:368-370); no valid pair: NaN
  const double mx = bits ? __longlong_as_double((long long)bits) : __longlong_as_double(0x7ff8000000000000LL);
  const long long C = f.C;
  for (int k = sub; k < unit.count; k += 1 << p.lane_shift) {
    const long long slot = unit.slot0 + k;
    const long long i = unit.col, j = unit.j_explicit ? f.pj_list[slot] : unit.j0 + k;
    const long long a = j + i * C, b = i + j * C;
    const int st = f.status[slot];
    if (st != 0) {
      // degenerate pair: the reference returns four NA (src/kendallc.cpp:193-199,225-244,292-298).  R's
      // NA_real_ is the NaN with low word 1954; written as bits so that an R binder needs no fix-up
      // pass over the matrices (a genuine NaN, e.g. the p-value of a two-row pair, stays a NaN)
      const double na = __longlong_as_double(0x7ff00000000007a2LL);
#pragma unroll
      for (int q = 0; q < 5; ++q)
        if (f.m[q]) { f.m[q][a] = na; f.m[q][b] = na; }
      atomicAdd(f.hist + (st & 15), 1ULL);  // degenerate pairs are rare
      continue;
    }
    const double raw = f.tau[slot];
    if (f.m[0]) { const double v = f.scale_max ? raw / mx : raw; f.m[0][a] = v; f.m[0][b] = v; }
    if (f.m[1]) { f.m[1][a] = raw; f.m[1][b] = raw; }
    if (f.m[2]) { const double v = f.pvalue[slot]; f.m[2][a] = v; f.m[2][b] = v; }
    if (f.m[3]) { const double v = f.taumax[slot]; f.m[3][a] = v; f.m[3][b] = v; }
    if (f.m[4]) { const double v = f.completeness[slot]; f.m[4][a] = v; f.m[4][b] = v; }
  }
}

// diag_good (R/kendalltau.R:374-386): raw = cor = n_good / max(n_good), pvalue 0, taumax 1,
// completeness n_good / n; appended after the scaling, so never scaled.  One CTA.
__global__ void __launch_bounds__(1024) matrix_diag_kernel(const MatrixFill f) {
  __shared__ int red[32];
  int best = 0;
  for (long long c = threadIdx.x; c < f.C; c += 1024) {
    const int g = f.n_good ? f.n_good[c] : (int)f.n - f.stats[c].n_na;
    best = max(best, g);
  }
#pragma unroll
  for (int d = 16; d >= 1; d >>= 1) best = max(best, __shfl_xor_sync(FULL, best, d));
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = best;
  __syncthreads();
  best = red[threadIdx.x & 31];
#pragma unroll
  for (int d = 16; d >= 1; d >>= 1) best = max(best, __shfl_xor_sync(FULL, best, d));
  for (long long c = threadIdx.x; c < f.C; c += 1024) {
    const int g = f.n_good ? f.n_good[c] : (int)f.n - f.stats[c].n_na;
    const double v = (double)g / (double)best;
    const long long d = c + c * f.C;
    if (f.m[0]) f.m[0][d] = v;
    if (f.m[1]) f.m[1][d] = v;
    if (f.m[2]) f.m[2][d] = 0.0;
    if (f.m[3]) f.m[3][d] = 1.0;
    if (f.m[4]) f.m[4][d] = (double)g / (double)f.n;
  }
}

// One warp per 32 rows of one column: a ballot is the mask word.
__global__ void __launch_bounds__(256) missing_bits_kernel(const double* __restrict__ data, long long ld, long long n,
                                                           long long C, const double* __restrict__ lit, int nlit,
                                                           int na_nan, int na_inf, uint32_t* __restrict__ bits,
                                                           long long words) {
  const long long col = blockIdx.x;
  const long long w = (long long)blockIdx.y * 8 + (threadIdx.x >> 5);
  if (w >= words) return;
  const long long r = w * 32 + (threadIdx.x & 31);
  bool miss = false;
  if (r < n) {
    const double v = data[col * ld + r];
    miss = (na_nan && v != v) || (na_inf && isinf(v));
    for (int g = 0; g < nlit; ++g) miss = miss || (v == lit[g]);
  }
  const unsigned word = __ballot_sync(FULL, miss);
  if ((threadIdx.x & 31) == 0) bits[w * C + col] = word;
}

// pair index -> (i, j) in utils::combn(C, 2) order, the diagonal appended
__device__ __forceinline__ void pair_of_index(long long C, long long index, long long& i, long long& j) {
  const long long ptri = C * (C - 1) / 2;
  if (index >= ptri) {
    i = j = index - ptri;
    return;
  }
  const double b = 2.0 * (double)C - 1.0;
  long long r = (long long)((b - sqrt(b * b - 8.0 * (double)index)) * 0.5);
  r = max(0LL, min(r, C - 2));
  while (r > 0 && r * (2 * C - r - 1) / 2 > index) --r;
  while (r + 1 < C - 1 && (r + 1) * (2 * C - r - 2) / 2 <= index) ++r;
  i = r;
  j = r + 1 + (index - r * (2 * C - r - 1) / 2);
}

__global__ void __launch_bounds__(256) pair_missing_kernel(const uint32_t* __restrict__ bits, long long words,
                                                           long long n, long long C, const int32_t* __restrict__ pi,
                                                           const int32_t* __restrict__ pj, long long P,
                                                           int32_t* __restrict__ missing,
                                                           double* __restrict__ completeness) {
  const long long p = (long long)blockIdx.x * 256 + threadIdx.x;
  if (p >= P) return;
  long long i, j;
  if (pi) {
    i = pi[p];
    j = pj[p];
  } else {
    pair_of_index(C, p, i, j);
  }
  int cnt = 0;
  for (long long w = 0; w < words; ++w) cnt += __popc(bits[w * C + i] | bits[w * C + j]);  // sum(in_x | in_y), :626
  if (missing) missing[p] = cnt;
  if (completeness) completeness[p] = 1.0 - (double)cnt / (double)n;  // :617
}

// full symmetric matrix, one thread per entry (the diagonal is a pair like any other: diag_good = FALSE, :586)
__global__ void __launch_bounds__(256) missing_matrix_kernel(const uint32_t* __restrict__ bits, long long words,
                                                             long long n, long long C, double* __restrict__ m) {
  const long long i = (long long)blockIdx.x * 256 + threadIdx.x, j = blockIdx.y;
  if (i >= C) return;
  int cnt = 0;
  for (long long w = 0; w < words; ++w) cnt += __popc(bits[w * C + i] | bits[w * C + j]);
  m[i + j * C] = 1.0 - (double)cnt / (double)n;
}

// CSC input -> dense columns [c_lo, c_lo + gridDim.x) of `out` (ld = n), one CTA per column: the CTA zero-fills
// its column with 16-byte stores (a column that starts on an odd element writes that one alone), then, after a
// barrier, scatters the column's stored entries.  rowidx / values are read coalesced; the rows of a column are
// sorted, so the scattered writes of a warp mostly fall into a few segments.
__global__ void __launch_bounds__(512) csc_expand_kernel(const int64_t* __restrict__ colptr,
                                                         const int32_t* __restrict__ rowidx,
                                                         const double* __restrict__ values, long long n,
                                                         long long c_lo, double* __restrict__ out) {
  const long long c = c_lo + blockIdx.x;
  double* col = out + c * n;
  const long long head = (reinterpret_cast<uintptr_t>(col) & 15) ? 1 : 0;
  const long long pairs = (n - head) >> 1;
  double2* body = reinterpret_cast<double2*>(col + head);
  for (long long k = threadIdx.x; k < pairs; k += blockDim.x) body[k] = make_double2(0.0, 0.0);
  if (threadIdx.x == 0 && head) col[0] = 0.0;
  if (threadIdx.x == 0 && head + 2 * pairs < n) col[n - 1] = 0.0;
  __syncthreads();
  const long long e = colptr[c + 1];
  for (long long k = colptr[c] + threadIdx.x; k < e; k += blockDim.x) col[rowidx[k]] = values[k];
}

// Multi-GPU matrix output: this device fills columns [c_lo, c_hi) of the five C x C matrices -- a
// contiguous block of every (column-major) matrix, so that it leaves for the caller's arrays as one
// copy per matrix.  The value of entry (r, c) is the result of pair (min, max) wherever that pair was
// computed: the per-pair result arrays of all devices are read in place (peer memory over NVLink, or
// the same device).  Rows below the diagonal of a column are consecutive pairs (coalesced reads), rows
// above it are one pair per row of the triangle (8-byte gathers; ~C^2/2 of them per job, a few MB over
// the links).  One thread per entry; writes are coalesced.
__global__ void __launch_bounds__(256) matrix_block_fill_kernel(const BlockFill f) {
  const long long r = (long long)blockIdx.x * 256 + threadIdx.x;
  const long long c = f.c_lo + blockIdx.y;
  if (r >= f.C) return;
  const long long C = f.C, ptri = C * (C - 1) / 2;
  const long long o = r + (c - f.c_lo) * C;
  const double na = __longlong_as_double(0x7ff00000000007a2LL);  // R's NA_real_
  long long k;
  if (r == c) {
    if (f.diag_good) {  // R/kendalltau.R:374-386, never scaled
      const double g = (double)f.n_good[c];
      if (f.m[0]) f.m[0][o] = g / (double)f.best_good;
      if (f.m[1]) f.m[1][o] = g / (double)f.best_good;
      if (f.m[2]) f.m[2][o] = 0.0;
      if (f.m[3]) f.m[3][o] = 1.0;
      if (f.m[4]) f.m[4][o] = g / (double)f.n;
      return;
    }
    k = ptri + c;  // the (i,i) pairs are computed pairs when !diag_good (R/kendalltau.R:191-194)
  } else {
    const long long i = r < c ? r : c, j = r < c ? c : r;
    k = i * (2 * C - i - 1) / 2 + (j - i - 1);
  }
  int d = 0;
  while (d + 1 < f.n_dev && k >= f.pair_lo[d + 1]) ++d;
  const long long slot = k - f.pair_lo[d];
  const int st = f.status[d][slot];
  const bool once = r >= c;  // every pair is met twice (both triangles): count it where r > c
  if (st != 0) {
#pragma unroll
    for (int q = 0; q < 5; ++q)
      if (f.m[q]) f.m[q][o] = na;
    if (once) atomicAdd(f.hist + (st & 15), 1ULL);
    return;
  }
  const double raw = f.tau[d][slot];
  if (f.m[0]) f.m[0][o] = f.scale_max ? raw / f.max_taumax : raw;
  if (f.m[1]) f.m[1][o] = raw;
  if (f.m[2]) f.m[2][o] = f.pvalue[d][slot];
  if (f.m[3]) f.m[3][o] = f.taumax[d][slot];
  if (f.m[4]) f.m[4][o] = f.completeness[d][slot];
}

}  // namespace

int launch_matrix_block_fill(const BlockFill& f, cudaStream_t stream) {
  const long long ncols = f.c_hi - f.c_lo;
  if (ncols <= 0) return 0;
  if (ncols > 65535) return -1;  // gridDim.y
  const dim3 grid((unsigned)((f.C + 255) / 256), (unsigned)ncols);
  matrix_block_fill_kernel<<<grid, 256, 0, stream>>>(f);
  return launch_status(1);
}

int launch_matrix_fill(const MatrixFill& mf, cudaStream_t stream) {
  int launches = 0;
  if (mf.n_units > 0) {
    FillParams p;
    p.f = mf;
    p.lane_shift = 0;
    while ((1 << p.lane_shift) < mf.max_unit_pairs && p.lane_shift < 5) ++p.lane_shift;
    const long long grid = ((mf.n_units << p.lane_shift) + 127) / 128;
    matrix_fill_kernel<<<(unsigned)grid, 128, 0, stream>>>(p);
    ++launches;
  }
  if (mf.diag_good) {
    matrix_diag_kernel<<<1, 1024, 0, stream>>>(mf);
    ++launches;
  }
  return launch_status(launches);
}

int launch_missing_bits(const double* d_data, int64_t ld, int64_t n, int64_t C, const double* d_lit, int nlit,
                        int na_nan, int na_inf, uint32_t* bits, int64_t words, cudaStream_t stream) {
  const dim3 grid((unsigned)C, (unsigned)((words + 7) / 8));
  missing_bits_kernel<<<grid, 256, 0, stream>>>(d_data, ld, n, C, d_lit, nlit, na_nan, na_inf, bits, words);
  return launch_status(1);
}

int launch_pair_missing(const uint32_t* bits, int64_t words, int64_t n, int64_t C, const int32_t* pi,
                        const int32_t* pj, int64_t P, int32_t* missing, double* completeness,
                        cudaStream_t stream) {
  if (P <= 0) return 0;
  pair_missing_kernel<<<(unsigned)((P + 255) / 256), 256, 0, stream>>>(bits, words, n, C, pi, pj, P, missing,
                                                                        completeness);
  return launch_status(1);
}

int launch_missing_matrix(const uint32_t* bits, int64_t words, int64_t n, int64_t C, double* matrix,
                          cudaStream_t stream) {
  if (C > 65535) return -1;  // gridDim.y
  const dim3 grid((unsigned)((C + 255) / 256), (unsigned)C);
  missing_matrix_kernel<<<grid, 256, 0, stream>>>(bits, words, n, C, matrix);
  return launch_status(1);
}

int launch_csc_expand(const int64_t* colptr, const int32_t* rowidx, const double* values, int64_t n, int64_t c_lo,
                      int64_t c_hi, double* out, cudaStream_t stream) {
  if (c_hi <= c_lo) return 0;
  csc_expand_kernel<<<(unsigned)(c_hi - c_lo), 512, 0, stream>>>(colptr, rowidx, values, n, c_lo, out);
  return launch_status(1);
}

}  // namespace icikt
