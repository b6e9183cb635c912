// icikt_padj.cu -- R's p.adjust on the device (icikt_padj.cuh has the arithmetic and why it is exact):
//   * padj_candidates: per window of a filtered call, the count of non-NaN p-values and the keys of those <= a bound,
//     appended to a candidate buffer.  The buffer is sorted before it is read, so the order in which the warps append
//     does not matter: one atomic per warp and window, no scan.
//   * padj_sort_scan: the radix sort of the candidates (CUB, from the toolkit's CCCL), the value of every sorted
//     position, and the running max (holm, bonferroni) or min (hochberg, BH, BY) over them.  Max and min are exact,
//     so CUB's parallel scan order gives the bits of R's sequential cummax / cummin.
//   * padj_lookup: a row's adjusted value, found by an upper-bound binary search of its p-value in the sorted keys.
//   * padj_array: the whole of p.adjust on a device array (icikt_p_adjust).
#include <algorithm>
#include <chrono>

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include "icikt_internal.h"
#include "icikt_padj.cuh"

namespace icikt {

namespace {

constexpr unsigned FULL = 0xffffffffu;
constexpr int kPadjThreads = 256;
constexpr unsigned long long kNanKey = ~0ull;  // above every non-NaN key: NaN p-values sort last

unsigned grid_for(int64_t n) {
  const int64_t blocks = (n + kPadjThreads - 1) / kPadjThreads;
  return (unsigned)std::min<int64_t>(std::max<int64_t>(blocks, 1), 148 * 16);
}

// counts[0] += non-NaN p-values, keys[counts[1]++] = every p <= bound (NaN bound: every non-NaN p)
__global__ void padj_candidate_kernel(const double* __restrict__ p, long long n,
                                                                      double bound, unsigned long long* counts,
                                                                      unsigned long long* __restrict__ keys) {
  const int lane = threadIdx.x & 31;
  const long long stride = (long long)gridDim.x * blockDim.x;
  unsigned long long valid = 0;
  // every lane of a warp runs the same number of rounds, so the ballots see the whole warp
  for (long long base = (long long)blockIdx.x * blockDim.x + (threadIdx.x & ~31); base < n; base += stride) {
    const long long k = base + lane;
    const double v = k < n ? p[k] : __longlong_as_double(0x7ff8000000000000LL);
    const bool ok = v == v;
    const bool cand = ok && (bound != bound || v <= bound);
    valid += ok;
    const unsigned word = __ballot_sync(FULL, cand);
    if (word) {
      unsigned long long at = 0;
      if (lane == 0) at = atomicAdd(counts + 1, (unsigned long long)__popc(word));
      at = __shfl_sync(FULL, at, 0);
      if (cand) keys[at + __popc(word & ((1u << lane) - 1u))] = padj_key(v);
    }
  }
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) valid += __shfl_down_sync(FULL, valid, d);
  if (lane == 0 && valid) atomicAdd(counts, valid);
}

// vals[s] = the value of sorted position i, s = i (scan up) or K - 1 - i (scan down, so that the scan runs forward)
__global__ void __launch_bounds__(kPadjThreads) padj_value_kernel(const unsigned long long* __restrict__ keys,
                                                                  long long K, long long m, int method, double q,
                                                                  double* __restrict__ vals) {
  const bool up = padj_scan_up(method);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < K; i += (long long)gridDim.x * blockDim.x) {
    const double v = padj_rank_value(method, m, i + 1, __longlong_as_double((long long)keys[i]), q);
    vals[up ? i : K - 1 - i] = v;
  }
}

// out[r] = pmin(1, value of the last sorted position whose key is <= p[r]'s); every p[r] is one of the keys
__global__ void __launch_bounds__(kPadjThreads) padj_lookup_kernel(const unsigned long long* __restrict__ keys,
                                                                   const double* __restrict__ vals, long long K,
                                                                   int method, const double* __restrict__ p,
                                                                   long long R, double* __restrict__ out) {
  const bool up = padj_scan_up(method);
  for (long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x; r < R; r += (long long)gridDim.x * blockDim.x) {
    const unsigned long long key = padj_key(p[r]);
    long long lo = 0, hi = K;  // first position whose key is > key
    while (lo < hi) {
      const long long mid = (lo + hi) >> 1;
      if (keys[mid] <= key) lo = mid + 1; else hi = mid;
    }
    const long long pos = lo - 1;
    out[r] = pos < 0 ? __longlong_as_double(0x7ff8000000000000LL) : padj_pmin1(vals[up ? pos : K - 1 - pos]);
  }
}

// p.adjust on an array: the (key, index) pairs to sort, NaN p-values under kNanKey; counts[0] += non-NaN values
__global__ void __launch_bounds__(kPadjThreads) padj_array_keys_kernel(const double* __restrict__ p, long long m,
                                                                       unsigned long long* __restrict__ keys,
                                                                       long long* __restrict__ idx,
                                                                       unsigned long long* counts) {
  unsigned long long valid = 0;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (long long)gridDim.x * blockDim.x) {
    const double v = p[i];
    keys[i] = v == v ? padj_key(v) : kNanKey;
    idx[i] = i;
    valid += v == v;
  }
  for (int d = 16; d > 0; d >>= 1) valid += __shfl_down_sync(FULL, valid, d);
  if ((threadIdx.x & 31) == 0 && valid) atomicAdd(counts, valid);
}

// out[idx[i]] = the adjusted value of sorted position i; the NaN p-values (positions >= mm) keep their bits
__global__ void __launch_bounds__(kPadjThreads) padj_array_scatter_kernel(const long long* __restrict__ idx,
                                                                          const double* __restrict__ vals, long long m,
                                                                          long long mm, int method,
                                                                          const double* __restrict__ p,
                                                                          double* __restrict__ out) {
  const bool up = padj_scan_up(method);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (long long)gridDim.x * blockDim.x) {
    const long long to = idx[i];
    out[to] = i < mm ? padj_pmin1(vals[up ? i : mm - 1 - i]) : p[to];
  }
}

struct MaxOp {
  __device__ double operator()(double a, double b) const { return a > b ? a : b; }
};
struct MinOp {
  __device__ double operator()(double a, double b) const { return a < b ? a : b; }
};

cudaError_t scan_vals(double* vals, int64_t K, int method, cudaStream_t stream) {
  size_t bytes = 0;
  cudaError_t e = padj_scan_up(method) ? cub::DeviceScan::InclusiveScan(nullptr, bytes, vals, MaxOp(), K, stream)
                                       : cub::DeviceScan::InclusiveScan(nullptr, bytes, vals, MinOp(), K, stream);
  if (e != cudaSuccess) return e;
  void* tmp = nullptr;
  if ((e = cudaMalloc(&tmp, std::max<size_t>(bytes, 1))) != cudaSuccess) return e;
  e = padj_scan_up(method) ? cub::DeviceScan::InclusiveScan(tmp, bytes, vals, MaxOp(), K, stream)
                           : cub::DeviceScan::InclusiveScan(tmp, bytes, vals, MinOp(), K, stream);
  const cudaError_t s = cudaStreamSynchronize(stream);
  cudaFree(tmp);
  return e != cudaSuccess ? e : s;
}

}  // namespace

cudaError_t padj_candidates(const double* p, int64_t n, double bound, unsigned long long* counts,
                            unsigned long long* keys, cudaStream_t stream) {
  if (n <= 0) return cudaSuccess;
  padj_candidate_kernel<<<grid_for(n), kPadjThreads, 0, stream>>>(p, n, bound, counts, keys);
  return cudaGetLastError();
}

cudaError_t padj_sort_scan(unsigned long long* keys, unsigned long long* alt, int64_t K, int64_t m, int method,
                           double q, unsigned long long** sorted, double** vals, cudaStream_t stream) {
  cub::DoubleBuffer<unsigned long long> db(keys, alt);
  size_t bytes = 0;
  cudaError_t e = cub::DeviceRadixSort::SortKeys(nullptr, bytes, db, K, 0, 63, stream);  // bit 63 is 0 in every key
  if (e != cudaSuccess) return e;
  void* tmp = nullptr;
  if ((e = cudaMalloc(&tmp, std::max<size_t>(bytes, 1))) != cudaSuccess) return e;
  e = cub::DeviceRadixSort::SortKeys(tmp, bytes, db, K, 0, 63, stream);
  const cudaError_t s = cudaStreamSynchronize(stream);
  cudaFree(tmp);
  if (e != cudaSuccess || s != cudaSuccess) return e != cudaSuccess ? e : s;
  *sorted = db.Current();
  *vals = reinterpret_cast<double*>(db.Alternate());
  padj_value_kernel<<<grid_for(K), kPadjThreads, 0, stream>>>(*sorted, K, m, method, q, *vals);
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  return scan_vals(*vals, K, method, stream);
}

cudaError_t padj_lookup(const unsigned long long* sorted, const double* vals, int64_t K, int method, const double* p,
                        int64_t R, double* out, cudaStream_t stream) {
  if (R <= 0) return cudaSuccess;
  padj_lookup_kernel<<<grid_for(R), kPadjThreads, 0, stream>>>(sorted, vals, K, method, p, R, out);
  return cudaGetLastError();
}

cudaError_t padj_array(const double* p, int64_t m, int method, double* out, int64_t* n_tests, double* q_ms,
                       cudaStream_t stream) {
  unsigned long long* keys[2] = {nullptr, nullptr};
  long long* idx[2] = {nullptr, nullptr};
  unsigned long long* counts = nullptr;
  void* tmp = nullptr;
  cudaError_t e = cudaSuccess;
  auto run = [&]() -> cudaError_t {
    for (int b = 0; b < 2; ++b) {
      if ((e = cudaMalloc(&keys[b], sizeof(unsigned long long) * (size_t)m)) != cudaSuccess) return e;
      if ((e = cudaMalloc(&idx[b], sizeof(long long) * (size_t)m)) != cudaSuccess) return e;
    }
    if ((e = cudaMalloc(&counts, sizeof(unsigned long long))) != cudaSuccess) return e;
    if ((e = cudaMemsetAsync(counts, 0, sizeof(unsigned long long), stream)) != cudaSuccess) return e;
    padj_array_keys_kernel<<<grid_for(m), kPadjThreads, 0, stream>>>(p, m, keys[0], idx[0], counts);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    cub::DoubleBuffer<unsigned long long> dk(keys[0], keys[1]);
    cub::DoubleBuffer<long long> di(idx[0], idx[1]);
    size_t bytes = 0;
    if ((e = cub::DeviceRadixSort::SortPairs(nullptr, bytes, dk, di, m, 0, 64, stream)) != cudaSuccess) return e;
    if ((e = cudaMalloc(&tmp, std::max<size_t>(bytes, 1))) != cudaSuccess) return e;
    if ((e = cub::DeviceRadixSort::SortPairs(tmp, bytes, dk, di, m, 0, 64, stream)) != cudaSuccess) return e;
    unsigned long long mm = 0;
    if ((e = cudaMemcpyAsync(&mm, counts, sizeof(mm), cudaMemcpyDeviceToHost, stream)) != cudaSuccess) return e;
    if ((e = cudaStreamSynchronize(stream)) != cudaSuccess) return e;
    *n_tests = (int64_t)mm;
    if (mm <= 1) return cudaMemcpyAsync(out, p, sizeof(double) * (size_t)m, cudaMemcpyDeviceToDevice, stream);
    const auto t0 = std::chrono::steady_clock::now();
    const double q = method == kPadjBY ? padj_by_q((int64_t)mm) : 0.0;
    if (q_ms) *q_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    double* vals = reinterpret_cast<double*>(dk.Alternate());
    padj_value_kernel<<<grid_for((int64_t)mm), kPadjThreads, 0, stream>>>(dk.Current(), (long long)mm, (long long)mm,
                                                                          method, q, vals);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    if ((e = scan_vals(vals, (int64_t)mm, method, stream)) != cudaSuccess) return e;
    padj_array_scatter_kernel<<<grid_for(m), kPadjThreads, 0, stream>>>(di.Current(), vals, m, (long long)mm, method,
                                                                        p, out);
    return cudaGetLastError();
  };
  e = run();
  const cudaError_t s = cudaStreamSynchronize(stream);
  for (int b = 0; b < 2; ++b) {
    cudaFree(keys[b]);
    cudaFree(idx[b]);
  }
  cudaFree(counts);
  cudaFree(tmp);
  return e != cudaSuccess ? e : s;
}

}  // namespace icikt
