// icikt_capi.cu -- host side of libicikt_b200.so: the C ABI declared in include/icikt_b200.h.
// Owns device memory, the streams, the pair-unit table and the CUDA-event timings; all
// arithmetic lives in icikt_columns.cu / icikt_pairs.cu.  There is no CPU fallback.
// Large all-pairs jobs of the one-shot entry points are pipelined (build_stage_table, run_staged):
// column chunks upload behind the pair launches of earlier chunks, finished row blocks of the
// results leave behind later ones.
#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <memory>
#include <mutex>
#include <new>
#include <string>
#include <condition_variable>
#include <thread>
#include <vector>

#include "../../include/icikt_b200.h"
#include "icikt_components.cuh"
#include "icikt_cross.cuh"
#include "icikt_edges.cuh"
#include "icikt_internal.h"
#include "icikt_owned.h"
#include "icikt_padj.cuh"
#include "icikt_topk.cuh"

using namespace icikt;

namespace {

thread_local std::string g_err;

int fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}
int cuda_fail(cudaError_t e, const char* what) {
  g_err = std::string(what) + ": " + cudaGetErrorString(e);
  return ICIKT_ERR_CUDA;
}
// failure of one of the launchers in icikt_columns.cu / icikt_pairs.cu / icikt_reshape.cu
int launch_fail(const char* what) {
  cudaError_t e = g_launch_error;
  if (e == cudaSuccess) e = cudaGetLastError();
  g_err = std::string(what) + ": " + (g_launch_note ? g_launch_note : "") + ": " + cudaGetErrorString(e);
  g_launch_error = cudaSuccess;
  g_launch_note = "";
  return ICIKT_ERR_CUDA;
}
#define CK(call)                                         \
  do {                                                   \
    cudaError_t e_ = (call);                             \
    if (e_ != cudaSuccess) return cuda_fail(e_, #call);  \
  } while (0)

// CK for the calls that allocate: running out of memory is ICIKT_ERR_ALLOC
#define ECK(call)                                                                                              \
  do {                                                                                                         \
    cudaError_t e_ = (call);                                                                                   \
    if (e_ != cudaSuccess)                                                                                     \
      return e_ == cudaErrorMemoryAllocation ? (cudaGetLastError(), fail(ICIKT_ERR_ALLOC, "allocation failed: " #call)) \
                                             : cuda_fail(e_, #call);                                           \
  } while (0)

// room for `count` elements in `a`, and `view` (a table the kernels take as a plain pointer) on it
template <typename T>
cudaError_t reserve_view(DeviceArray<T>& a, T*& view, size_t count) {
  const cudaError_t e = a.reserve(count);
  view = a.get();
  return e;
}

int64_t tri_pairs(int64_t C) { return C * (C - 1) / 2; }
int64_t row_start(int64_t i, int64_t C) { return i * (2 * C - i - 1) / 2; }

}  // namespace

// result sets up to stage_all() bytes: one pinned copy of everything; above: two pinned chunks of
// stage_chunk() bytes (the environment overrides exist for the tests)
static size_t env_bytes(const char* name, size_t dflt) {
  const char* e = std::getenv(name);
  const long long v = e ? std::atoll(e) : 0;
  return v > 0 ? (size_t)v : dflt;
}
static size_t stage_all() { return env_bytes("ICIKT_STAGE_ALL", 96u << 20); }
static size_t stage_chunk() { return env_bytes("ICIKT_STAGE_CHUNK", 32u << 20); }

// One launch of the pipelined one-shot call.
struct StageLaunch {
  int64_t col_lo = 0, col_hi = 0;    // columns uploaded and preprocessed right before it (empty: none)
  int64_t unit_lo = 0, unit_hi = 0;  // its units
  int64_t slot_lo = 0, slot_hi = 0;  // results complete once it has run: a contiguous range of the pair order
  int max_unit_pairs = 1;
};

// The launches of the pipelined one-shot call over all pairs of C columns (combn order, then the C diagonal
// pairs if include_diag).  Columns arrive in chunks [0, f), [f, 2f), [2f, 4f) ... (f ~ C/16): the launch of a
// chunk covers every pair (i, j), i < j, whose LATER column j lies in the chunk, so it needs nothing that has
// not been uploaded, and the upload of the next chunk hides behind it (the work of a chunk grows with the
// square of the columns, the upload linearly).  The last chunk holds most of the pairs; it is cut into
// `n_blocks` row blocks of about equal work: once the block of rows [r0, r1) has run, every pair of those rows
// is done -- slots [row_start(r0), row_start(r1)) of the pair order -- and can be copied out while the next
// block runs.  Units never straddle rows; their length tapers off towards the end of a launch (long units
// while much work is left, single pairs at the end) so that the persistent CTAs run dry together.
void build_stage_table(int64_t C, bool include_diag, int64_t cta_slots, int n_blocks, std::vector<PairUnit>& U,
                       std::vector<StageLaunch>& S) {
  U.clear();
  S.clear();
  const int64_t ptri = C * (C - 1) / 2;
  auto rstart = [C](int64_t i) { return i * (2 * C - i - 1) / 2; };
  std::vector<int64_t> cb{0};
  int64_t f = std::max<int64_t>(64, ((C / 16) + 7) & ~int64_t(7));
  for (; 4 * f <= 3 * C; f *= 2) cb.push_back(f);
  cb.push_back(C);
  // pairs (i, j) with r0 <= i < r1 and max(i + 1, lo) <= j < hi, as units appended to U
  auto emit = [&](int64_t r0, int64_t r1, int64_t lo, int64_t hi, StageLaunch& st) {
    int64_t total = 0;
    for (int64_t i = r0; i < r1; ++i) total += std::max<int64_t>(0, hi - std::max(i + 1, lo));
    const int64_t ulen_max = std::max<int64_t>(1, std::min<int64_t>(16, total / (16 * cta_slots)));
    int64_t left = total;
    st.unit_lo = (int64_t)U.size();
    for (int64_t i = r0; i < r1; ++i) {
      const int64_t ja = std::max(i + 1, lo);
      for (int64_t j = ja; j < hi;) {
        const int64_t want = std::max<int64_t>(1, std::min<int64_t>(ulen_max, left / (4 * cta_slots)));
        const int64_t len = std::min<int64_t>(want, hi - j);
        PairUnit u;
        u.slot0 = rstart(i) + (j - i - 1);
        u.col = (int32_t)i;
        u.j0 = (int32_t)j;
        u.count = (int32_t)len;
        u.j_explicit = 0;
        U.push_back(u);
        st.max_unit_pairs = std::max(st.max_unit_pairs, (int)len);
        j += len;
        left -= len;
      }
    }
    st.unit_hi = (int64_t)U.size();
  };
  const size_t nchunks = cb.size() - 1;
  for (size_t s = 0; s + 1 < nchunks; ++s) {
    StageLaunch st;
    st.col_lo = cb[s];
    st.col_hi = cb[s + 1];
    emit(0, cb[s + 1] - 1, cb[s], cb[s + 1], st);
    S.push_back(st);
  }
  // the last chunk in row blocks of about equal work
  const int64_t lo = cb[nchunks - 1];
  int64_t total = 0;
  for (int64_t i = 0; i + 1 < C; ++i) total += C - std::max(i + 1, lo);
  const int B = (int)std::max<int64_t>(1, std::min<int64_t>(n_blocks, total / std::max<int64_t>(1, 64 * cta_slots)));
  int64_t r0 = 0, acc = 0;
  for (int b = 0; b < B; ++b) {
    int64_t r1 = r0;
    const int64_t goal = total * (b + 1) / B;
    if (b == B - 1) {
      r1 = std::max<int64_t>(C - 1, 0);
      acc = total;
    } else {
      while (r1 + 1 < C && acc < goal) {
        acc += C - std::max(r1 + 1, lo);
        ++r1;
      }
    }
    StageLaunch st;
    if (b == 0) {
      st.col_lo = lo;
      st.col_hi = C;
    }
    emit(r0, r1, lo, C, st);
    st.slot_lo = rstart(r0);
    st.slot_hi = (b == B - 1) ? ptri : rstart(r1);
    if (b == B - 1 && include_diag) {
      for (int64_t i = 0; i < C; ++i) {
        PairUnit u;
        u.slot0 = ptri + i;
        u.col = (int32_t)i;
        u.j0 = (int32_t)i;
        u.count = 1;
        u.j_explicit = 0;
        U.push_back(u);
      }
      st.unit_hi = (int64_t)U.size();
      st.slot_hi = ptri + C;
    }
    S.push_back(st);
    r0 = r1;
  }
}

struct icikt_plan {
  int device = 0;
  int n_sm = 0;
  // the streams come before every buffer and event, so that those are released first
  Stream stream;
  Stream copy_stream;  // uploads and downloads of a staged run and of the window walk
  int64_t n = 0, C = 0, P = 0;
  icikt_opts opts{};
  bool want_counts = false;

  DeviceArray<double> d_data_own;
  const double* d_data = nullptr;
  int64_t ld = 0;
  DeviceArray<double> d_global_na;
  // CSC input (the *_csc entry points): the stored entries on the device, each at its global entry number;
  // csc_expand_kernel rebuilds d_data_own from them ahead of K1.  Kept with the plan, grown on demand.
  DeviceArray<int64_t> d_colptr;  // [C + 1]
  DeviceArray<int32_t> d_rowidx;
  DeviceArray<double> d_values;
  int64_t expand_lo = 0, expand_hi = 0;  // columns uploaded as CSC and not expanded yet
  int64_t expand_dst = 0;                // ... and the matrix column their column 0 lands on (cross calls: Y at Cx)

  // the column tables and the column path's scratch as the kernels take them, and the memory behind them
  ColumnTables tab;
  ColumnWork wk;
  struct {
    DeviceArray<uint16_t> perm, rank, trow, trun, tend, lgrp, gstart, vals_in;
    DeviceArray<uint32_t> tord, nabits, firstbits, gpos;
    DeviceArray<ColStats> stats;
    DeviceArray<int32_t> max_tied;
    DeviceArray<unsigned long long> keys_in, keys_out;
  } col_mem;
  bool columns_done = false;
  // launch shapes of the pair kernel, one per tier (see tiled_shape): no large tie groups /
  // large tie groups sorted in place / pass B.  All are enqueued; the device-side maxima over the
  // columns pick the one that runs (no host round trip).
  TiledShape shape, shape_mid, shape_heavy;
  DeviceArray<unsigned char> d_scratch;  // global-memory variant of the pair kernel

  std::vector<PairUnit> units;
  int max_unit_pairs = 1;  // longest unit
  DeviceArray<PairUnit> d_units;
  DeviceArray<int32_t> d_pj;
  DeviceArray<PairRaw> d_raw;
  DeviceArray<PairComplete> d_pw;  // complete-observations mode
  // results, packed in one allocation so that one copy brings them to the host:
  // [tau P][pvalue P][taumax P][completeness P] doubles, [max taumax bits] u64, [status P] int32
  DeviceArray<unsigned char> d_res;
  PinnedArray<unsigned char> h_res;  // pinned staging copy (small and medium result sets only)
  // staged copies (ensure_stage): two pinned chunks of stage_bytes, copy-out and uploads pipelined
  PinnedArray<unsigned char> h_stage[2];
  Event stage_ev[2];
  size_t stage_bytes = 0;
  bool stage_busy[2] = {false, false};  // an upload out of the chunk is in flight (staged_copy_in)
  double *d_tau = nullptr, *d_p = nullptr, *d_tm = nullptr, *d_comp = nullptr;
  unsigned long long* d_maxbits = nullptr;
  int32_t* d_status = nullptr;
  DeviceArray<int64_t> d_counts;
  DeviceArray<unsigned long long> d_scalars;  // [0] unit counter, [1] max taumax bits
  DeviceArray<unsigned char> d_naive;
  int64_t naive_threads = 0;
  // matrix output (ensure_matrix_buffers), allocated on first use
  DeviceArray<double> d_mat;          // 5 x [C][C]: cor, raw, pvalue, taumax, completeness (multi-GPU: 5 blocks of columns)
  PinnedArray<unsigned char> h_mat;   // pinned copy of all five (small C only)
  DeviceArray<unsigned long long> d_hist;  // [16] pairs per status class
  DeviceArray<int32_t> d_ngood;       // [C] caller-supplied n_good
  bool pairs_done = false;

  // Pipelined one-shot call (staged plans only, see build_stage_table / run_staged): the pair order is cut
  // into launches that need only the columns uploaded so far, then into row blocks whose results are
  // contiguous in the pair order and leave while the next block is computed.
  bool staged = false;
  bool staged_run = false;               // the last run went through run_staged (selects the timing sums)
  std::vector<StageLaunch> stages;
  std::vector<Event> sync_ev;            // per launch: [2l] its columns have landed, [2l+1] its results are ready
  std::vector<Event> time_ev;            // per launch: K1 start/end, K2 start, K2 end, K3 end

  // Filtered all-pairs call (icikt_all_pairs_edges, see run_edges): the plan's pair buffers hold one window of
  // the pair order; units, selected rows and the per-window readback are double-buffered.
  DeviceArray<PairUnit> d_wunits[2];
  PinnedArray<PairUnit> h_wunits[2];
  DeviceArray<uint32_t> d_emask;
  DeviceArray<uint32_t> d_etile;
  DeviceArray<EdgeRow> d_erows[2];
  DeviceArray<unsigned long long> d_etotal;  // [2]
  PinnedArray<unsigned long long> h_estat;   // [2][2]: rows kept, max taumax bits so far
  Event eev[2][6];                           // per buffer: units up start/end, K2 start, K2 end, K3 end, selection end
  // Top-k all-pairs call (icikt_all_pairs_topk), on the same window walk: per-column candidate counts, the
  // candidates of one window, and the lists of the L columns that keep one (all C, or one side of a cross call)
  DeviceArray<uint32_t> d_tcount;  // [L]
  DeviceArray<uint2> d_tcand;      // [2 W]
  DeviceArray<TopkCol> d_tcol;     // [L]
  DeviceArray<int32_t> d_tidx;     // [L k]
  DeviceArray<double> d_tlist;     // 4 x [L k]: raw, pvalue, taumax, completeness
  // Cross per-pair call (icikt_cross_pairs): a window's results, moved off the pair buffers so that they can be
  // copied out while the next window runs; [tau W][pvalue W][taumax W][completeness W] doubles, [status W] int32
  DeviceArray<unsigned char> d_cres[2];
  // Top-k over several devices (icikt_all_pairs_topk_multi): this device's block of columns of the merged lists
  DeviceArray<int32_t> d_mn;     // [C] entries kept per column of the block
  DeviceArray<int32_t> d_midx;   // [entries]
  DeviceArray<double> d_mlist;   // 4 x [entries]: raw, pvalue, taumax, completeness
  // Edge-count calls (icikt_all_pairs_count_edges), summed over the windows: [16] pairs per status class, [T] passing
  // pairs per filter, then, if degrees are wanted, [T][C] degrees (filter-major), then, for the component calls, [T]
  // successful hooks; d_eparent holds their [T][C] union-find forests (icikt_components.cuh)
  DeviceArray<unsigned long long> d_ecount;
  DeviceArray<int32_t> d_eparent;

  Event ev[9];
  icikt_timings tm{};

  // A failed call may leave copies in flight: none may still read a caller's array once the plan is gone.  The
  // handles then release themselves on the plan's device.
  ~icikt_plan() {
    cudaSetDevice(device);
    if (copy_stream) cudaStreamSynchronize(copy_stream);
    if (stream) cudaStreamSynchronize(stream);
    cudaGetLastError();
  }
};

namespace {

// The units of pairs [lo, hi) of the all-pairs order of C columns (combn order, then the diagonal if
// include_diag), appended to U with slots counted from lo.  `first_row`: a row at or before the row of pair lo
// (0 always works; the filtered call passes the row of its window).
void range_units(int64_t C, bool include_diag, int64_t lo, int64_t hi, int64_t slots, std::vector<PairUnit>& U,
                 int64_t first_row = 0) {
  const int64_t ptri = tri_pairs(C);
  int64_t ulen = (hi - lo) / (16 * slots);
  ulen = std::max<int64_t>(1, std::min<int64_t>(16, ulen));
  for (int64_t i = first_row; i + 1 < C; ++i) {
    const int64_t rs = row_start(i, C), re = rs + (C - 1 - i);
    const int64_t a = std::max(rs, lo), b = std::min(re, hi);
    for (int64_t s = a; s < b; s += ulen) {
      PairUnit u;
      u.slot0 = s - lo;
      u.col = (int32_t)i;
      u.j0 = (int32_t)(i + 1 + (s - rs));
      u.count = (int32_t)std::min<int64_t>(ulen, b - s);
      u.j_explicit = 0;
      U.push_back(u);
    }
    if (re >= hi) break;
  }
  if (include_diag) {
    for (int64_t i = std::max<int64_t>(0, lo - ptri); i < C; ++i) {
      const int64_t s = ptri + i;
      if (s < lo || s >= hi) continue;
      PairUnit u;
      u.slot0 = s - lo;
      u.col = (int32_t)i;
      u.j0 = (int32_t)i;
      u.count = 1;
      u.j_explicit = 0;
      U.push_back(u);
    }
  }
}

// Split the pair order into units: consecutive pairs that share their first column.
int build_units(icikt_plan* p, const int32_t* pi, const int32_t* pj, int64_t P_list) {
  const int64_t C = p->C;
  std::vector<PairUnit>& U = p->units;
  U.clear();
  const int64_t slots = (int64_t)p->n_sm * 2;
  if (!pi) {
    const int64_t ptot = tri_pairs(C) + (p->opts.include_diag ? C : 0);
    int64_t lo = p->opts.pair_lo, hi = p->opts.pair_hi;
    if (lo == 0 && hi == 0) hi = ptot;
    if (lo < 0 || hi > ptot || lo > hi) return fail(ICIKT_ERR_BAD_ARG, "pair_lo/pair_hi out of range");
    p->P = hi - lo;
    range_units(C, p->opts.include_diag != 0, lo, hi, slots, U);
  } else {
    p->P = P_list;
    for (int64_t k = 0; k < P_list; ++k)
      if (pi[k] < 0 || pi[k] >= C || pj[k] < 0 || pj[k] >= C)
        return fail(ICIKT_ERR_BAD_ARG, "pair index out of range");
    int64_t ulen = P_list / (16 * slots);
    ulen = std::max<int64_t>(1, std::min<int64_t>(16, ulen));
    int64_t k = 0;
    while (k < P_list) {
      int64_t e = k + 1;
      while (e < P_list && e - k < ulen && pi[e] == pi[k]) ++e;
      PairUnit u;
      u.slot0 = k;
      u.col = pi[k];
      u.j0 = pj[k];
      u.count = (int32_t)(e - k);
      u.j_explicit = 1;
      U.push_back(u);
      k = e;
    }
  }
  return ICIKT_OK;
}

int select_device(int device) {
  int cnt = 0;
  if (cudaGetDeviceCount(&cnt) != cudaSuccess || cnt < 1) {
    cudaGetLastError();
    return fail(ICIKT_ERR_NO_DEVICE, "no CUDA device available (this library has no CPU fallback)");
  }
  if (device < 0 || device >= cnt) return fail(ICIKT_ERR_BAD_ARG, "device ordinal out of range");
  CK(cudaSetDevice(device));
  return ICIKT_OK;
}

// memcpy into the caller's (usually freshly allocated, not yet faulted-in) array: one thread moves
// about 5 GB/s there, a PCIe 5 link delivers ten times that, so large blocks are split over a few
// threads (ICIKT_COPY_THREADS, default min(8, hardware threads); 1 = plain memcpy)
int copy_threads() {
  static const int n_threads = [] {
    const char* e = std::getenv("ICIKT_COPY_THREADS");
    int t = e ? std::atoi(e) : (int)std::min(8u, std::max(1u, std::thread::hardware_concurrency()));
    return std::max(1, std::min(t, 64));
  }();
  return n_threads;
}

void host_copy(void* dst, const void* src, size_t bytes) {
  const int n_threads = copy_threads();
  constexpr size_t kMinPart = 2u << 20;
  const int parts = (int)std::min<size_t>((size_t)n_threads, bytes / kMinPart);
  if (parts <= 1) {
    std::memcpy(dst, src, bytes);
    return;
  }
  const size_t per = ((bytes / parts) + 4095) & ~size_t(4095);
  std::vector<std::thread> th;
  th.reserve((size_t)parts - 1);
  for (int k = 1; k < parts; ++k) {
    const size_t o = per * k;
    if (o >= bytes) break;
    const size_t l = std::min(per, bytes - o);
    th.emplace_back([=] { std::memcpy(static_cast<unsigned char*>(dst) + o, static_cast<const unsigned char*>(src) + o, l); });
  }
  std::memcpy(dst, src, std::min(per, bytes));
  for (auto& t : th) t.join();
}

// Device -> pageable host memory through two pinned chunks: the copy of chunk k+1 runs while chunk k
// is moved from the staging buffer into the caller's array (cudaMemcpyAsync straight into pageable
// memory is staged by the driver at a fraction of the link rate).
int staged_copy_out(icikt_plan* p, void* dst, const void* d_src, size_t bytes, cudaStream_t stream) {
  unsigned char* out = static_cast<unsigned char*>(dst);
  const unsigned char* src = static_cast<const unsigned char*>(d_src);
  size_t off[2] = {0, 0}, len[2] = {0, 0};
  int k = 0;
  p->stage_busy[0] = p->stage_busy[1] = false;  // uploads out of the chunks precede these copies in stream order
  for (size_t o = 0; o < bytes || len[0] || len[1]; ++k) {
    const int cur = k & 1;
    if (len[cur]) {  // the chunk issued two steps ago has landed in h_stage[cur]
      CK(cudaEventSynchronize(p->stage_ev[cur]));
      host_copy(out + off[cur], p->h_stage[cur].get(), len[cur]);
      len[cur] = 0;
    }
    if (o < bytes) {
      const size_t l = std::min(p->stage_bytes, bytes - o);
      CK(cudaMemcpyAsync(p->h_stage[cur].get(), src + o, l, cudaMemcpyDeviceToHost, stream));
      CK(cudaEventRecord(p->stage_ev[cur], stream));
      off[cur] = o;
      len[cur] = l;
      o += l;
    }
  }
  return ICIKT_OK;
}

// the two pinned chunks of the staged copies and their events (kept with the plan)
int ensure_stage(icikt_plan* p) {
  if (!p->stage_bytes) p->stage_bytes = stage_chunk();
  for (int i = 0; i < 2; ++i) {
    ECK(p->h_stage[i].reserve(p->stage_bytes));
    if (!p->stage_ev[i]) ECK(p->stage_ev[i].create(cudaEventDisableTiming));
  }
  return ICIKT_OK;
}

// Pageable host memory -> device through the plan's two pinned chunks: cudaMemcpyAsync from pageable
// memory is staged by the driver on one thread (~10 GB/s, a fraction of the link); here chunk k + 1 is
// copied into pinned memory by several host threads while chunk k is on the wire.  The source is fully
// consumed when this returns (same guarantee as the plain call).
int staged_copy_in(icikt_plan* p, void* d_dst, const void* src, size_t bytes, cudaStream_t stream) {
  int rc = ensure_stage(p);
  if (rc != ICIKT_OK) return rc;
  unsigned char* dst = static_cast<unsigned char*>(d_dst);
  const unsigned char* in = static_cast<const unsigned char*>(src);
  int k = 0;
  for (size_t o = 0; o < bytes; ++k) {
    const int cur = k & 1;
    if (p->stage_busy[cur]) {  // the chunk sent two steps ago (possibly by the previous call) has left
      CK(cudaEventSynchronize(p->stage_ev[cur]));
      p->stage_busy[cur] = false;
    }
    const size_t l = std::min(p->stage_bytes, bytes - o);
    host_copy(p->h_stage[cur].get(), in + o, l);
    CK(cudaMemcpyAsync(dst + o, p->h_stage[cur].get(), l, cudaMemcpyHostToDevice, stream));
    CK(cudaEventRecord(p->stage_ev[cur], stream));
    p->stage_busy[cur] = true;
    o += l;
  }
  return ICIKT_OK;
}

bool host_is_pinned(const void* ptr) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, ptr) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return a.type == cudaMemoryTypeHost || a.type == cudaMemoryTypeManaged;
}

// Where the columns of a call come from: a dense column-major matrix (data, ld) or a CSC matrix (colptr
// [C + 1], rowidx / values [colptr[C]], checked by check_csc) of C columns (icikt_input of the public header).
struct ColumnSource {
  int64_t C = 0;
  const double* data = nullptr;
  int64_t ld = 0;
  const int64_t* colptr = nullptr;
  const int32_t* rowidx = nullptr;
  const double* values = nullptr;
  bool csc() const { return colptr != nullptr; }
};
ColumnSource dense_source(const double* data, int64_t ld, int64_t C) {
  ColumnSource s;
  s.C = C;
  s.data = data;
  s.ld = ld;
  return s;
}
ColumnSource csc_source(const int64_t* colptr, const int32_t* rowidx, const double* values, int64_t C) {
  ColumnSource s;
  s.C = C;
  s.colptr = colptr;
  s.rowidx = rowidx;
  s.values = values;
  return s;
}

// first column of [c_lo, c_hi) with a row outside [0, n) or rows that do not strictly increase; c_hi if none
int64_t first_bad_column(const int64_t* colptr, const int32_t* rowidx, int64_t n, int64_t c_lo, int64_t c_hi) {
  for (int64_t c = c_lo; c < c_hi; ++c) {
    int64_t prev = -1;
    for (int64_t k = colptr[c]; k < colptr[c + 1]; ++k) {
      const int64_t r = rowidx[k];
      if (r < 0 || r >= n || r <= prev) return c;
      prev = r;
    }
  }
  return c_hi;
}

// The host-side checks of a CSC matrix, before any device work: colptr starts at 0 and never decreases, the
// arrays exist if there are entries, and the rows of every column lie in [0, n) and strictly increase.  The
// row scan of a large matrix is split over a few host threads (ICIKT_COPY_THREADS, as the copies); the
// message names the first bad column either way.
int check_csc(const int64_t* colptr, const int32_t* rowidx, const double* values, int64_t n, int64_t C) {
  if (n < 1 || C < 1) return fail(ICIKT_ERR_BAD_ARG, "n and C must be >= 1");
  if (!colptr) return fail(ICIKT_ERR_BAD_ARG, "CSC input: colptr is NULL");
  if (colptr[0] != 0) return fail(ICIKT_ERR_BAD_ARG, "CSC input: colptr[0] is " + std::to_string(colptr[0]) + ", not 0");
  for (int64_t c = 0; c < C; ++c)
    if (colptr[c + 1] < colptr[c])
      return fail(ICIKT_ERR_BAD_ARG, "CSC input: colptr decreases at column " + std::to_string(c) + " (" +
                                         std::to_string(colptr[c]) + " -> " + std::to_string(colptr[c + 1]) + ")");
  const int64_t nnz = colptr[C];
  if (nnz > 0 && (!rowidx || !values))
    return fail(ICIKT_ERR_BAD_ARG, "CSC input: colptr[C] = " + std::to_string(nnz) +
                                       " entries but rowidx or values is NULL");
  const int parts = (int)std::min<int64_t>(std::min<int64_t>(copy_threads(), C), nnz >> 20);
  int64_t bad = C;
  if (parts <= 1) {
    bad = first_bad_column(colptr, rowidx, n, 0, C);
  } else {  // column ranges of about equal entry counts
    std::vector<int64_t> lo((size_t)parts + 1, C), found((size_t)parts, C);
    lo[0] = 0;
    for (int t = 1; t < parts; ++t)
      lo[(size_t)t] = std::upper_bound(colptr, colptr + C + 1, nnz * t / parts) - colptr - 1;
    std::vector<std::thread> th;
    for (int t = 1; t < parts; ++t)
      th.emplace_back([&, t] { found[(size_t)t] = first_bad_column(colptr, rowidx, n, lo[(size_t)t], lo[(size_t)t + 1]); });
    found[0] = first_bad_column(colptr, rowidx, n, 0, lo[1]);
    for (auto& x : th) x.join();
    for (int t = 0; t < parts; ++t)
      if (found[(size_t)t] < lo[(size_t)t + 1]) { bad = found[(size_t)t]; break; }
  }
  if (bad == C) return ICIKT_OK;
  int64_t prev = -1;
  for (int64_t k = colptr[bad];; ++k) {  // first_bad_column stopped inside this column
    const int64_t r = rowidx[k];
    if (r < 0 || r >= n)
      return fail(ICIKT_ERR_BAD_ARG, "CSC input: row " + std::to_string(r) + " of column " + std::to_string(bad) +
                                         " is outside [0, " + std::to_string(n) + ")");
    if (r <= prev)
      return fail(ICIKT_ERR_BAD_ARG, "CSC input: rows of column " + std::to_string(bad) +
                                         (r == prev ? " repeat row " + std::to_string(r)
                                                    : " are not sorted (" + std::to_string(prev) + " before " +
                                                          std::to_string(r) + ")"));
    prev = r;
  }
}

// host -> device copy of a contiguous array; pageable memory of 8 MB and more goes through the plan's pinned
// chunks (staged_copy_in), as a dense matrix does
int copy_array_in(icikt_plan* p, void* d_dst, const void* src, size_t bytes, cudaStream_t stream) {
  if (bytes == 0) return ICIKT_OK;
  if (bytes >= (8u << 20) && !std::getenv("ICIKT_NO_STAGED_UPLOAD") && !host_is_pinned(src))
    return staged_copy_in(p, d_dst, src, bytes, stream);
  CK(cudaMemcpyAsync(d_dst, src, bytes, cudaMemcpyHostToDevice, stream));
  return ICIKT_OK;
}

// CSC columns [c_lo, c_hi): the colptr slice and the slices [colptr[c_lo], colptr[c_hi]) of rowidx and values,
// on `stream`.  The columns are expanded into d_data_own (source column c at matrix column dst + c) by the next
// plan_columns_impl or expand_columns, on the compute stream.
// (Neighbouring chunks of a pipelined call both copy their shared colptr entry; the second copy writes the
// value the expansion of the first chunk may be reading.)
int copy_csc_in(icikt_plan* p, const ColumnSource& s, int64_t c_lo, int64_t c_hi, int64_t dst, cudaStream_t stream) {
  const int64_t nnz = s.colptr[s.C];
  CK(p->d_colptr.reserve((size_t)p->C + 1));
  if (nnz > 0) {  // nothing of an earlier call is in flight: every call ends with its streams idle
    CK(p->d_rowidx.reserve((size_t)nnz));
    CK(p->d_values.reserve((size_t)nnz));
  }
  p->expand_lo = p->expand_hi = 0;
  if (c_hi <= c_lo) return ICIKT_OK;
  const int64_t k_lo = s.colptr[c_lo], k_hi = s.colptr[c_hi];
  CK(cudaMemcpyAsync(p->d_colptr.get() + c_lo, s.colptr + c_lo, sizeof(int64_t) * (size_t)(c_hi - c_lo + 1),
                     cudaMemcpyHostToDevice, stream));
  int rc = copy_array_in(p, p->d_rowidx.get() + k_lo, s.rowidx + k_lo, sizeof(int32_t) * (size_t)(k_hi - k_lo), stream);
  if (rc == ICIKT_OK)
    rc = copy_array_in(p, p->d_values.get() + k_lo, s.values + k_lo, sizeof(double) * (size_t)(k_hi - k_lo), stream);
  if (rc != ICIKT_OK) return rc;
  p->expand_lo = c_lo;
  p->expand_hi = c_hi;
  p->expand_dst = dst;
  return ICIKT_OK;
}

// host -> device copy of columns [c_lo, c_hi) of `s` into the plan's own matrix buffer at matrix columns
// [dst + c_lo, dst + c_hi) (CSC: of their stored entries), on `stream`
int copy_columns_in(icikt_plan* p, const ColumnSource& s, int64_t c_lo, int64_t c_hi, cudaStream_t stream,
                    int64_t dst = 0) {
  CK(p->d_data_own.reserve((size_t)p->n * p->C));
  if (s.csc()) return copy_csc_in(p, s, c_lo, c_hi, dst, stream);
  p->expand_lo = p->expand_hi = 0;
  const double* data = s.data;
  const int64_t ld = s.ld;
  if (c_hi <= c_lo) return ICIKT_OK;
  double* out = p->d_data_own.get() + (size_t)(dst + c_lo) * p->n;
  const size_t bytes = sizeof(double) * (size_t)p->n * (size_t)(c_hi - c_lo);
  if (ld == p->n && bytes >= (8u << 20) && !std::getenv("ICIKT_NO_STAGED_UPLOAD") && !host_is_pinned(data + (size_t)c_lo * ld))
    return staged_copy_in(p, out, data + (size_t)c_lo * ld, bytes, stream);
  CK(cudaMemcpy2DAsync(out, sizeof(double) * p->n, data + (size_t)c_lo * ld,
                       sizeof(double) * ld, sizeof(double) * p->n, (size_t)(c_hi - c_lo), cudaMemcpyHostToDevice, stream));
  return ICIKT_OK;
}

int upload_columns(icikt_plan* p, const ColumnSource& s, int64_t c_lo, int64_t c_hi) {
  CK(cudaSetDevice(p->device));
  CK(cudaEventRecord(p->ev[0], p->stream));
  const int rc = copy_columns_in(p, s, c_lo, c_hi, p->stream);
  if (rc != ICIKT_OK) return rc;
  CK(cudaEventRecord(p->ev[1], p->stream));
  p->d_data = p->d_data_own.get();
  p->ld = p->n;
  p->columns_done = false;
  p->pairs_done = false;
  p->staged_run = false;
  return ICIKT_OK;
}

// reusable barrier for the worker threads of icikt_all_pairs_multi
class HostBarrier {
 public:
  explicit HostBarrier(int n) : n_(n) {}
  void wait() {
    std::unique_lock<std::mutex> lk(mu_);
    const int gen = gen_;
    if (++count_ == n_) {
      count_ = 0;
      ++gen_;
      cv_.notify_all();
    } else {
      cv_.wait(lk, [&] { return gen != gen_; });
    }
  }

 private:
  std::mutex mu_;
  std::condition_variable cv_;
  int n_, count_ = 0, gen_ = 0;
};

// the matrix fill's buffers (kept with the plan): `elems` doubles of matrices (`what` names them in the error), the
// status histogram and n_good
int ensure_matrix_buffers(icikt_plan* p, size_t elems, const char* what) {
  if (p->d_mat.reserve(elems) != cudaSuccess) {
    cudaGetLastError();
    return fail(ICIKT_ERR_ALLOC, std::string("device allocation of ") + what + " failed");
  }
  CK(p->d_hist.reserve(16));
  CK(p->d_ngood.reserve((size_t)p->C));
  return ICIKT_OK;
}

// elapsed time between two completed events; 0 if one of them was never recorded
float ev_ms(cudaEvent_t a, cudaEvent_t b) {
  float ms = 0.f;
  if (cudaEventElapsedTime(&ms, a, b) != cudaSuccess) ms = 0.f;
  return ms;
}

}  // namespace

extern "C" {

void icikt_default_opts(icikt_opts* o) {
  if (!o) return;
  std::memset(o, 0, sizeof(*o));
  o->perspective = ICIKT_PERSPECTIVE_GLOBAL;
  o->alternative = ICIKT_ALT_TWO_SIDED;
  o->kernel = ICIKT_KERNEL_TILED;
}

int icikt_abi_version(void) { return ICIKT_ABI_VERSION; }

int icikt_device_count(void) {
  int cnt = 0;
  if (cudaGetDeviceCount(&cnt) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return cnt;
}

int64_t icikt_max_n(void) { return tiled_max_n(); }

const char* icikt_last_error(void) { return g_err.c_str(); }

// `staged`: the unit table of the pipelined one-shot call (all pairs only), see build_stage_table
static int plan_create_impl(icikt_plan** out, int64_t n, int64_t C, const int32_t* pi, const int32_t* pj,
                            int64_t P, const icikt_opts* opts_in, bool staged) {
  if (!out) return fail(ICIKT_ERR_BAD_ARG, "plan pointer is NULL");
  *out = nullptr;
  if (n < 1 || C < 1) return fail(ICIKT_ERR_BAD_ARG, "n and C must be >= 1");
  if ((pi == nullptr) != (pj == nullptr)) return fail(ICIKT_ERR_BAD_ARG, "pi and pj must both be given");
  if (pi && P < 1) return fail(ICIKT_ERR_BAD_ARG, "empty pair list");
  if (n > tiled_max_n()) return fail(ICIKT_ERR_TOO_LONG, "n exceeds icikt_max_n()");
  if (C > 2147483647LL) return fail(ICIKT_ERR_BAD_ARG, "too many columns");
  icikt_opts o;
  if (opts_in) o = *opts_in; else icikt_default_opts(&o);
  int rc = select_device(o.device);
  if (rc != ICIKT_OK) return rc;

  std::unique_ptr<icikt_plan> p(new (std::nothrow) icikt_plan());
  if (!p) return fail(ICIKT_ERR_ALLOC, "out of host memory");
  p->device = o.device;
  p->opts = o;
  p->want_counts = o.want_counts != 0;
  p->n = n;
  p->C = C;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, o.device) != cudaSuccess) return fail(ICIKT_ERR_CUDA, "cudaGetDeviceProperties failed");
  p->n_sm = prop.multiProcessorCount;
  if (prop.major < 10)
    return fail(ICIKT_ERR_NO_DEVICE, "device is not sm_100-class; this library is built for sm_100a only");
  if (staged) {
    if (pi || o.pair_lo != 0 || o.pair_hi != 0) return fail(ICIKT_ERR_BAD_ARG, "staged plans cover all pairs");
    p->staged = true;
    p->P = tri_pairs(C) + (o.include_diag ? C : 0);
    // row blocks of the last chunk: the copy-out of the final block is all that stays exposed
    int blocks = (size_t)p->P * (4 * sizeof(double) + sizeof(int32_t)) > stage_all() ? 16 : 8;
    if (const char* e = std::getenv("ICIKT_PIPELINE_BLOCKS")) blocks = std::max(1, std::min(64, std::atoi(e)));
    build_stage_table(C, o.include_diag != 0, (int64_t)p->n_sm * 2, blocks, p->units, p->stages);
  } else {
    rc = build_units(p.get(), pi, pj, P);
    if (rc != ICIKT_OK) return rc;
  }
  for (const PairUnit& u : p->units) p->max_unit_pairs = std::max(p->max_unit_pairs, (int)u.count);

  ECK(p->stream.create());
  for (Event& e : p->ev) ECK(e.create());
  if (staged) {
    ECK(p->copy_stream.create());
    p->sync_ev.resize(2 * p->stages.size());
    p->time_ev.resize(5 * p->stages.size());
    for (Event& e : p->sync_ev) ECK(e.create(cudaEventDisableTiming));
    for (Event& e : p->time_ev) ECK(e.create());
  }
  ColumnTables& t = p->tab;
  auto& m = p->col_mem;
  t.n = n;
  t.C = C;
  t.nstride = (n + 63) & ~63LL;
  const int64_t nwords = ((n + 31) & ~31LL) / 32;
  t.wstride = (nwords + 3) & ~3LL;
  const size_t ne = (size_t)t.nstride * C, nw = (size_t)t.wstride * C;
  ECK(reserve_view(m.perm, t.perm, ne));
  ECK(reserve_view(m.rank, t.rank, ne));
  ECK(reserve_view(m.trow, t.trow, ne));
  ECK(reserve_view(m.trun, t.trun, ne));
  ECK(reserve_view(m.tend, t.tend, ne));
  ECK(reserve_view(m.tord, t.tord, ne));
  ECK(reserve_view(m.nabits, t.nabits, nw));
  ECK(reserve_view(m.firstbits, t.firstbits, nw));
  t.gstride = t.nstride + 64;
  ECK(reserve_view(m.gstart, t.gstart, (size_t)t.gstride * C));
  ECK(reserve_view(m.lgrp, t.lgrp, (size_t)kLargeStride * C));
  ECK(reserve_view(m.stats, t.stats, (size_t)C));
  ECK(reserve_view(m.max_tied, t.max_tied, 4));
  // padding words of the bit arrays (beyond n32/32) are never written by the kernels
  ECK(cudaMemsetAsync(t.nabits, 0, sizeof(uint32_t) * nw, p->stream));
  ECK(cudaMemsetAsync(t.firstbits, 0, sizeof(uint32_t) * nw, p->stream));
  ECK(cudaMemsetAsync(t.max_tied, 0, 4 * sizeof(int32_t), p->stream));
  p->shape = tiled_shape(n, 0, t.wstride, p->n_sm);
  if (!columns_fused(n)) {  // scratch of the multi-kernel column path (long columns)
    ECK(reserve_view(m.keys_in, p->wk.keys_in, ne));
    ECK(reserve_view(m.keys_out, p->wk.keys_out, ne));
    ECK(reserve_view(m.vals_in, p->wk.vals_in, ne));
    ECK(reserve_view(m.gpos, p->wk.gpos, (size_t)(t.nstride + 64) * C));
  }
  ECK(p->d_global_na.reserve(64));

  const size_t np = (size_t)std::max<int64_t>(p->P, 1);
  ECK(p->d_units.reserve(p->units.size()));
  ECK(cudaMemcpyAsync(p->d_units.get(), p->units.data(), sizeof(PairUnit) * p->units.size(),
                      cudaMemcpyHostToDevice, p->stream));
  if (pi) {
    ECK(p->d_pj.reserve(np));
    ECK(cudaMemcpyAsync(p->d_pj.get(), pj, sizeof(int32_t) * np, cudaMemcpyHostToDevice, p->stream));
  }
  ECK(p->d_raw.reserve(np));
  if (o.perspective == ICIKT_PERSPECTIVE_COMPLETE) ECK(p->d_pw.reserve(np));
  const size_t res_bytes = np * (4 * sizeof(double) + sizeof(int32_t)) + sizeof(unsigned long long);
  ECK(p->d_res.reserve(res_bytes));
  p->d_tau = reinterpret_cast<double*>(p->d_res.get());
  p->d_p = p->d_tau + np;
  p->d_tm = p->d_p + np;
  p->d_comp = p->d_tm + np;
  p->d_maxbits = reinterpret_cast<unsigned long long*>(p->d_comp + np);
  p->d_status = reinterpret_cast<int32_t*>(p->d_maxbits + 1);
  if (res_bytes <= stage_all()) {
    ECK(p->h_res.reserve(res_bytes));
  } else {
    rc = ensure_stage(p.get());
    if (rc != ICIKT_OK) return rc;
  }
  if (p->want_counts) ECK(p->d_counts.reserve(np * ICIKT_NCOUNTS));
  ECK(p->d_scalars.reserve(2));  // [0] unit counter
  if (o.kernel == ICIKT_KERNEL_NAIVE) {
    p->naive_threads = std::min<int64_t>((int64_t)p->units.size(), (int64_t)p->n_sm * 256);
    p->naive_threads = std::max<int64_t>(p->naive_threads, 1);
    ECK(p->d_naive.reserve(naive_scratch_bytes(n, p->naive_threads)));
  }
  ECK(cudaStreamSynchronize(p->stream));  // pj / units are read from caller memory
  *out = p.release();
  return ICIKT_OK;
}

int icikt_plan_create(icikt_plan** out, int64_t n, int64_t C, const int32_t* pi, const int32_t* pj,
                      int64_t P, const icikt_opts* opts_in) {
  return plan_create_impl(out, n, C, pi, pj, P, opts_in, false);
}

int64_t icikt_plan_num_pairs(const icikt_plan* p) { return p ? p->P : 0; }

int icikt_plan_upload(icikt_plan* p, const double* data, int64_t ld) {
  if (!p || !data || ld < p->n) return fail(ICIKT_ERR_BAD_ARG, "bad upload arguments");
  return upload_columns(p, dense_source(data, ld, p->C), 0, p->C);
}

int icikt_plan_set_device_matrix(icikt_plan* p, const double* d_data, int64_t ld) {
  if (!p || !d_data || ld < p->n) return fail(ICIKT_ERR_BAD_ARG, "bad device matrix arguments");
  p->d_data = d_data;
  p->ld = ld;
  p->expand_lo = p->expand_hi = 0;
  p->columns_done = false;
  p->pairs_done = false;
  CK(cudaSetDevice(p->device));
  CK(cudaEventRecord(p->ev[0], p->stream));
  CK(cudaEventRecord(p->ev[1], p->stream));
  return ICIKT_OK;
}

// the CSC columns uploaded and not expanded yet, expanded into d_data_own on the plan's stream; returns the
// launches or < 0 (the error is set)
static int expand_columns(icikt_plan* p) {
  if (p->expand_hi <= p->expand_lo) return 0;
  const int l = launch_csc_expand(p->d_colptr.get(), p->d_rowidx.get(), p->d_values.get(), p->n, p->expand_lo, p->expand_hi,
                                  p->d_data_own.get() + (size_t)p->expand_dst * p->n, p->stream);
  if (l < 0) return launch_fail("CSC expansion kernel"), -1;
  p->expand_lo = p->expand_hi = p->expand_dst = 0;
  return l;
}

// K1 over columns [col_lo, col_hi); `finish`: the statistics of every column are in place afterwards
// (a full run), so the pair kernel may be launched
// `reset`: a partial run that starts a sequence of partial runs over all columns on this device (the
// column kernels then raise the tier maxima themselves); e0/e1: timing events (default ev[2], ev[3])
static int plan_columns_impl(icikt_plan* p, const double* global_na, int32_t n_global_na, int64_t col_lo,
                             int64_t col_hi, bool finish, bool reset = false, cudaEvent_t e0 = nullptr,
                             cudaEvent_t e1 = nullptr) {
  if (!p || !p->d_data) return fail(ICIKT_ERR_BAD_ARG, "no matrix set on the plan");
  if (n_global_na < 0 || (n_global_na > 0 && !global_na)) return fail(ICIKT_ERR_BAD_ARG, "bad global_na");
  if (col_lo < 0 || col_hi > p->C || col_lo > col_hi) return fail(ICIKT_ERR_BAD_ARG, "column range out of bounds");
  CK(cudaSetDevice(p->device));
  // R/utils.R:6-15: NA and Inf entries of global_na select classes, the rest are literals
  double lit[64];
  int nlit = 0, na_inf = p->opts.na_inf;
  for (int i = 0; i < n_global_na; ++i) {
    const double v = global_na[i];
    if (std::isnan(v)) continue;
    if (std::isinf(v)) { na_inf = 1; continue; }
    if (nlit == 64) return fail(ICIKT_ERR_BAD_ARG, "more than 64 global_na literals");
    lit[nlit++] = v;
  }
  if (nlit) CK(cudaMemcpyAsync(p->d_global_na.get(), lit, sizeof(double) * nlit, cudaMemcpyHostToDevice, p->stream));
  if (reset) CK(cudaMemsetAsync(p->tab.max_tied, 0, 4 * sizeof(int32_t), p->stream));
  CK(cudaEventRecord(e0 ? e0 : p->ev[2], p->stream));
  // columns uploaded as CSC become dense first (their copies precede this point on the stream)
  const int expand_launches = expand_columns(p);
  if (expand_launches < 0) return ICIKT_ERR_CUDA;
  // the largest tier decides whether the global scratch may be needed at all
  const int64_t n_units = (int64_t)p->units.size();
  const bool inplace_ok = p->opts.perspective != ICIKT_PERSPECTIVE_COMPLETE;  // that mode has no in-place kernel
  p->shape = tiled_shape(p->n, 0, p->tab.wstride, p->n_sm, n_units, inplace_ok);
  p->shape_mid = tiled_shape(p->n, 1, p->tab.wstride, p->n_sm, n_units, inplace_ok);
  p->shape_heavy = tiled_shape(p->n, 2, p->tab.wstride, p->n_sm, n_units, inplace_ok);
  const TiledShape& worst = p->shape_heavy;
  const int slot_bytes = std::max(worst.region_bytes, worst.const_region_bytes);
  const int slot_ctas = std::max(std::max(worst.max_ctas, p->shape.max_ctas), std::max(p->shape_mid.max_ctas, p->n_sm * 2));
  const bool any_gmem = worst.gmem || worst.const_gmem || p->shape.gmem || p->shape_mid.gmem;
  const size_t need = (size_t)slot_ctas * (size_t)slot_bytes;
  if (any_gmem && need > p->d_scratch.size()) {
    // the shape depends on the perspective class and on tuning knobs in the environment, so a cached
    // plan may need a larger scratch than the one it was given first
    CK(cudaStreamSynchronize(p->stream));
    if (p->d_scratch.reserve(need) != cudaSuccess) {
      cudaGetLastError();
      return fail(ICIKT_ERR_ALLOC, "device allocation of the pair kernel's global scratch failed");
    }
  }
  for (TiledShape* sh : {&p->shape, &p->shape_mid, &p->shape_heavy}) {
    sh->scratch_stride = p->d_scratch ? slot_bytes : 0;
    sh->scratch_ctas = p->d_scratch ? (int)std::min<size_t>((size_t)slot_ctas, p->d_scratch.size() / (size_t)slot_bytes) : 0;
  }
  const int lc = launch_columns(p->d_data, p->ld, p->d_global_na.get(), nlit, na_inf, p->tab, p->wk, p->shape,
                                p->d_scratch.get(), p->stream, col_lo, col_hi);
  if (lc < 0) return launch_fail("column kernels");
  const int l = lc + expand_launches;
  CK(cudaEventRecord(e1 ? e1 : p->ev[3], p->stream));
  // no synchronisation: `lit` is pageable host memory, so the copy above was staged before
  // cudaMemcpyAsync returned
  p->tm.n_launches = reset || !e0 ? l : p->tm.n_launches + l;
  p->columns_done = finish;
  p->pairs_done = false;
  return ICIKT_OK;
}

int icikt_plan_columns(icikt_plan* p, const double* global_na, int32_t n_global_na) {
  if (!p) return fail(ICIKT_ERR_BAD_ARG, "plan is NULL");
  return plan_columns_impl(p, global_na, n_global_na, 0, p->C, true);
}

int icikt_plan_columns_range(icikt_plan* p, const double* global_na, int32_t n_global_na, int64_t col_lo,
                             int64_t col_hi) {
  if (!p) return fail(ICIKT_ERR_BAD_ARG, "plan is NULL");
  return plan_columns_impl(p, global_na, n_global_na, col_lo, col_hi, false);
}

int icikt_plan_columns_finish(icikt_plan* p) {
  if (!p || !p->d_data) return fail(ICIKT_ERR_BAD_ARG, "no matrix set on the plan");
  CK(cudaSetDevice(p->device));
  const int l = launch_max_tied(p->tab, p->stream);
  if (l < 0) return launch_fail("tier maxima kernel");
  CK(cudaEventRecord(p->ev[3], p->stream));  // the exchange of the tables counts as column time
  p->tm.n_launches += l;
  p->columns_done = true;
  return ICIKT_OK;
}

int icikt_plan_upload_columns(icikt_plan* p, const double* data, int64_t ld, int64_t col_lo, int64_t col_hi) {
  if (!p || !data || ld < p->n || col_lo < 0 || col_hi > p->C || col_lo > col_hi)
    return fail(ICIKT_ERR_BAD_ARG, "bad upload arguments");
  return upload_columns(p, dense_source(data, ld, p->C), col_lo, col_hi);
}

int icikt_plan_tables(icikt_plan* p, icikt_table* out, int32_t cap) {
  if (!p) return fail(ICIKT_ERR_BAD_ARG, "plan is NULL");
  const ColumnTables& t = p->tab;
  const bool complete = p->opts.perspective == ICIKT_PERSPECTIVE_COMPLETE;
  // the sorted positions of the tied rows are read only by the pair kernel's variants for long vectors
  // (rank table not staged: in place / global scratch)
  bool positions = false;
  for (int tier = 0; tier < 3; ++tier) {
    const TiledShape sh = tiled_shape(p->n, tier, t.wstride, p->n_sm, 0, !complete);
    positions = positions || sh.gmem || sh.inplace_kk != 0;
  }
  const icikt_table all[] = {
      {t.perm, (int64_t)(2 * t.nstride)},       {t.rank, (int64_t)(2 * t.nstride)},
      {t.trow, (int64_t)(2 * t.nstride)},       {t.trun, (int64_t)(2 * t.nstride)},
      {t.tord, (int64_t)(4 * t.nstride)},       {t.nabits, (int64_t)(4 * t.wstride)},
      {t.firstbits, (int64_t)(4 * t.wstride)},  {t.lgrp, (int64_t)(2 * kLargeStride)},
      {t.stats, (int64_t)sizeof(ColStats)},     {t.tend, (int64_t)(2 * t.nstride)},
      {t.gstart, (int64_t)(2 * t.gstride)},
  };
  int n_out = 0;
  for (const icikt_table& e : all) {
    if (e.ptr == (void*)t.tend && !positions) continue;
    if (e.ptr == (void*)t.gstart && !complete) continue;  // that mode only
    if (out && n_out < cap) out[n_out] = e;
    ++n_out;
  }
  return n_out;
}

// K2 (every tier's shape; the device-side maxima pick the one that runs) + K3 over units [unit_lo, unit_hi) of
// `units` (device; the plan's own table unless the filtered call passes a window's); e_start / e_mid / e_end
// bracket K2 and K3 on the plan's stream
static int launch_pair_group(icikt_plan* p, const PairUnit* units, int64_t unit_lo, int64_t unit_hi, int max_unit_pairs, cudaEvent_t e_start,
                             cudaEvent_t e_mid, cudaEvent_t e_end, int* launches_out) {
  CK(cudaMemsetAsync(p->d_scalars.get(), 0, 2 * sizeof(unsigned long long), p->stream));
  CK(cudaEventRecord(e_start, p->stream));
  PairLaunch pl;
  pl.tab = &p->tab;
  pl.units = units + unit_lo;
  pl.n_units = unit_hi - unit_lo;
  pl.pj_list = p->d_pj.get();
  pl.raw = p->d_raw.get();
  pl.pw = (p->opts.perspective == ICIKT_PERSPECTIVE_COMPLETE) ? p->d_pw.get() : nullptr;
  pl.unit_counter = p->d_scalars.get();
  pl.scratch = p->d_scratch.get();
  int launches = 0;
  if (pl.n_units <= 0) {
    CK(cudaEventRecord(e_mid, p->stream));
  } else {
    int l;
    if (pl.pw && p->opts.kernel == ICIKT_KERNEL_NAIVE)
      return fail(ICIKT_ERR_BAD_ARG, "the complete-observations mode needs the tiled kernel");
    if (p->opts.kernel == ICIKT_KERNEL_NAIVE)
      l = launch_pairs_naive(pl, p->P, reinterpret_cast<uint32_t*>(p->d_naive.get()), p->naive_threads, p->stream);
    else {
      l = launch_pairs_tiled(pl, p->shape, p->n_sm, 0, p->stream);
      if (l > 0) {
        const int l2 = launch_pairs_tiled(pl, p->shape_mid, p->n_sm, 1, p->stream);
        l = l2 < 0 ? l2 : l + l2;
      }
      if (l > 0) {
        const int l3 = launch_pairs_tiled(pl, p->shape_heavy, p->n_sm, 2, p->stream);
        l = l3 < 0 ? l3 : l + l3;
      }
    }
    if (l == -2)
      return fail(ICIKT_ERR_TOO_LONG, "the tied-value lists of this matrix do not fit the pair kernel's "
                                      "shared memory (long vectors with heavy ties)");
    if (l < 0) return launch_fail("pair kernel");
    launches += l;
    CK(cudaEventRecord(e_mid, p->stream));
    EpilogueLaunch el;
    el.tab = &p->tab;
    el.units = pl.units;
    el.n_units = pl.n_units;
    el.max_unit_pairs = max_unit_pairs;
    el.pj_list = p->d_pj.get();
    el.raw = p->d_raw.get();
    el.pw = pl.pw;
    el.perspective = p->opts.perspective;
    el.alternative = p->opts.alternative;
    el.continuity = p->opts.continuity;
    el.tau = p->d_tau;
    el.pvalue = p->d_p;
    el.taumax = p->d_tm;
    el.completeness = p->d_comp;
    el.status = p->d_status;
    el.counts = p->d_counts.get();
    el.max_taumax_bits = p->d_maxbits;
    l = launch_epilogue(el, p->stream);
    if (l < 0) return launch_fail("epilogue kernel");
    launches += l;
  }
  CK(cudaEventRecord(e_end, p->stream));
  *launches_out += launches;
  return ICIKT_OK;
}

int icikt_plan_pairs(icikt_plan* p) {
  if (!p || !p->columns_done) return fail(ICIKT_ERR_BAD_ARG, "icikt_plan_columns has not run");
  CK(cudaSetDevice(p->device));
  CK(cudaMemsetAsync(p->d_maxbits, 0, sizeof(unsigned long long), p->stream));
  int launches = 0;
  const int rc = launch_pair_group(p, p->d_units.get(), 0, (int64_t)p->units.size(), p->max_unit_pairs, p->ev[4], p->ev[8], p->ev[5], &launches);
  if (rc != ICIKT_OK) return rc;
  p->tm.n_launches = (p->tm.n_launches & 0xffff) | (launches << 16);
  p->pairs_done = true;
  p->staged_run = false;
  return ICIKT_OK;
}

int icikt_plan_sync(icikt_plan* p) {
  if (!p) return fail(ICIKT_ERR_BAD_ARG, "plan is NULL");
  CK(cudaSetDevice(p->device));
  CK(cudaStreamSynchronize(p->stream));
  return ICIKT_OK;
}

int icikt_plan_download(icikt_plan* p, double* raw, double* pvalue, double* taumax, double* completeness,
                        int32_t* status, int64_t* counts, double* max_taumax) {
  if (!p) return fail(ICIKT_ERR_BAD_ARG, "plan is NULL");
  if (counts && !p->d_counts) return fail(ICIKT_ERR_BAD_ARG, "plan was created without want_counts");
  CK(cudaSetDevice(p->device));
  const size_t np = (size_t)p->P;
  CK(cudaEventRecord(p->ev[6], p->stream));
  unsigned long long bits = 0;
  if (p->h_res) {
    // one device-to-host copy into pinned memory, then plain host copies into the caller's arrays
    CK(cudaMemcpyAsync(p->h_res.get(), p->d_res.get(), p->d_res.size(), cudaMemcpyDeviceToHost, p->stream));
    if (counts && np) CK(cudaMemcpyAsync(counts, p->d_counts.get(), sizeof(int64_t) * np * ICIKT_NCOUNTS, cudaMemcpyDeviceToHost, p->stream));
    CK(cudaEventRecord(p->ev[7], p->stream));
    CK(cudaStreamSynchronize(p->stream));
    const size_t npad = std::max<size_t>(np, 1);
    const double* h = reinterpret_cast<const double*>(p->h_res.get());
    if (np) {
      if (raw) host_copy(raw, h, sizeof(double) * np);
      if (pvalue) host_copy(pvalue, h + npad, sizeof(double) * np);
      if (taumax) host_copy(taumax, h + 2 * npad, sizeof(double) * np);
      if (completeness) host_copy(completeness, h + 3 * npad, sizeof(double) * np);
      if (status) host_copy(status, p->h_res.get() + 4 * npad * sizeof(double) + sizeof(unsigned long long), sizeof(int32_t) * np);
    }
    std::memcpy(&bits, h + 4 * npad, sizeof(bits));
  } else {
    if (np) {
      int rc = ICIKT_OK;
      if (raw) rc = staged_copy_out(p, raw, p->d_tau, sizeof(double) * np, p->stream);
      if (rc == ICIKT_OK && pvalue) rc = staged_copy_out(p, pvalue, p->d_p, sizeof(double) * np, p->stream);
      if (rc == ICIKT_OK && taumax) rc = staged_copy_out(p, taumax, p->d_tm, sizeof(double) * np, p->stream);
      if (rc == ICIKT_OK && completeness) rc = staged_copy_out(p, completeness, p->d_comp, sizeof(double) * np, p->stream);
      if (rc == ICIKT_OK && status) rc = staged_copy_out(p, status, p->d_status, sizeof(int32_t) * np, p->stream);
      if (rc == ICIKT_OK && counts) rc = staged_copy_out(p, counts, p->d_counts.get(), sizeof(int64_t) * np * ICIKT_NCOUNTS, p->stream);
      if (rc != ICIKT_OK) return rc;
    }
    CK(cudaMemcpyAsync(&bits, p->d_maxbits, sizeof(bits), cudaMemcpyDeviceToHost, p->stream));
    CK(cudaEventRecord(p->ev[7], p->stream));
    CK(cudaStreamSynchronize(p->stream));
  }
  if (max_taumax) {
    double v;
    std::memcpy(&v, &bits, sizeof(v));
    *max_taumax = bits ? v : std::nan("");
  }
  return ICIKT_OK;
}

int icikt_plan_download_matrices(icikt_plan* p, int32_t scale_max, int32_t diag_good, const int32_t* n_good,
                                 double* cor, double* raw, double* pvalue, double* taumax, double* completeness,
                                 int64_t* status_counts, double* max_taumax) {
  if (!p || !p->pairs_done) return fail(ICIKT_ERR_BAD_ARG, "icikt_plan_pairs has not run");
  CK(cudaSetDevice(p->device));
  const size_t C = (size_t)p->C, cc = C * C;
  double* outs[5] = {cor, raw, pvalue, taumax, completeness};
  int rc = ensure_matrix_buffers(p, 5 * cc, "the result matrices");
  if (rc != ICIKT_OK) return rc;
  CK(cudaEventRecord(p->ev[6], p->stream));
  // entries no pair writes stay 0 (R/kendalltau.R:389-396 start from matrix(0, ...)); with every pair
  // and the diagonal present nothing needs clearing
  const int64_t ptot = tri_pairs(p->C) + (p->opts.include_diag ? p->C : 0);
  const bool covered = !p->d_pj && p->P == ptot && (p->opts.include_diag || diag_good);
  MatrixFill mf{};
  for (int k = 0; k < 5; ++k) {
    mf.m[k] = outs[k] ? p->d_mat.get() + (size_t)k * cc : nullptr;
    if (outs[k] && !covered) CK(cudaMemsetAsync(mf.m[k], 0, sizeof(double) * cc, p->stream));
  }
  CK(cudaMemsetAsync(p->d_hist.get(), 0, 16 * sizeof(unsigned long long), p->stream));
  if (n_good) CK(cudaMemcpyAsync(p->d_ngood.get(), n_good, sizeof(int32_t) * C, cudaMemcpyHostToDevice, p->stream));
  mf.units = p->d_units.get();
  mf.n_units = (int64_t)p->units.size();
  mf.max_unit_pairs = p->max_unit_pairs;
  mf.pj_list = p->d_pj.get();
  mf.tau = p->d_tau;
  mf.pvalue = p->d_p;
  mf.taumax = p->d_tm;
  mf.completeness = p->d_comp;
  mf.status = p->d_status;
  mf.max_taumax_bits = p->d_maxbits;
  mf.stats = p->tab.stats;
  mf.n_good = n_good ? p->d_ngood.get() : nullptr;
  mf.n = p->n;
  mf.C = p->C;
  mf.scale_max = scale_max != 0;
  mf.diag_good = diag_good != 0;
  mf.hist = p->d_hist.get();
  if (p->P <= 0) mf.n_units = 0;
  if (launch_matrix_fill(mf, p->stream) < 0) return launch_fail("matrix fill kernel");
  const size_t all_bytes = 5 * cc * sizeof(double);
  if (all_bytes <= stage_all()) {
    CK(p->h_mat.reserve(all_bytes));
    for (int k = 0; k < 5; ++k)
      if (outs[k])
        CK(cudaMemcpyAsync(p->h_mat.get() + (size_t)k * cc * sizeof(double), mf.m[k], sizeof(double) * cc,
                           cudaMemcpyDeviceToHost, p->stream));
    CK(cudaStreamSynchronize(p->stream));
    for (int k = 0; k < 5; ++k)
      if (outs[k]) host_copy(outs[k], p->h_mat.get() + (size_t)k * cc * sizeof(double), sizeof(double) * cc);
  } else {
    rc = ensure_stage(p);
    for (int k = 0; k < 5 && rc == ICIKT_OK; ++k)
      if (outs[k]) rc = staged_copy_out(p, outs[k], mf.m[k], sizeof(double) * cc, p->stream);
    if (rc != ICIKT_OK) return rc;
  }
  unsigned long long hist[16], bits = 0;
  CK(cudaMemcpyAsync(hist, p->d_hist.get(), sizeof(hist), cudaMemcpyDeviceToHost, p->stream));
  CK(cudaMemcpyAsync(&bits, p->d_maxbits, sizeof(bits), cudaMemcpyDeviceToHost, p->stream));
  CK(cudaEventRecord(p->ev[7], p->stream));
  CK(cudaStreamSynchronize(p->stream));
  if (status_counts) {
    int64_t bad = 0;
    for (int k = 1; k < ICIKT_NSTATUS; ++k) { status_counts[k] = (int64_t)hist[k]; bad += status_counts[k]; }
    status_counts[0] = p->P - bad;
  }
  if (max_taumax) {
    double v;
    std::memcpy(&v, &bits, sizeof(v));
    *max_taumax = bits ? v : std::nan("");
  }
  return ICIKT_OK;
}

int icikt_plan_column_info(icikt_plan* p, int32_t* n_na) {
  if (!p || !p->columns_done) return fail(ICIKT_ERR_BAD_ARG, "icikt_plan_columns has not run");
  CK(cudaSetDevice(p->device));
  std::vector<ColStats> s((size_t)p->C);
  CK(cudaMemcpyAsync(s.data(), p->tab.stats, sizeof(ColStats) * s.size(), cudaMemcpyDeviceToHost, p->stream));
  CK(cudaStreamSynchronize(p->stream));
  if (n_na)
    for (int64_t c = 0; c < p->C; ++c) n_na[c] = s[(size_t)c].n_na;
  return ICIKT_OK;
}

void* icikt_plan_stream(icikt_plan* p) { return p ? (void*)p->stream : nullptr; }

int icikt_plan_timings(icikt_plan* p, icikt_timings* t) {
  if (!p || !t) return fail(ICIKT_ERR_BAD_ARG, "NULL argument");
  CK(cudaSetDevice(p->device));
  CK(cudaStreamSynchronize(p->stream));
  const int launches = (p->tm.n_launches & 0xffff) + (p->tm.n_launches >> 16);
  std::memset(t, 0, sizeof(*t));
  t->n_launches = launches;
  if (p->copy_stream) CK(cudaStreamSynchronize(p->copy_stream));
  // the streams are idle, so every recorded event has completed
  t->h2d_ms = ev_ms(p->ev[0], p->ev[1]);
  if (p->staged_run) {
    // pipelined call: kernel times are sums over the launches; h2d = start until the last column has landed,
    // d2h = first result copy until the last one (both overlap the kernels, so the parts exceed total_ms)
    for (size_t l = 0; l < p->stages.size(); ++l) {
      const Event* e = &p->time_ev[5 * l];
      if (p->stages[l].col_hi > p->stages[l].col_lo) t->columns_ms += ev_ms(e[0], e[1]);
      t->pairs_ms += ev_ms(e[2], e[3]);
      t->epilogue_ms += ev_ms(e[3], e[4]);
    }
  } else {
    t->columns_ms = ev_ms(p->ev[2], p->ev[3]);
    t->pairs_ms = ev_ms(p->ev[4], p->ev[8]);
    t->epilogue_ms = ev_ms(p->ev[8], p->ev[5]);
  }
  t->d2h_ms = ev_ms(p->ev[6], p->ev[7]);
  t->total_ms = ev_ms(p->ev[0], p->ev[7]);
  cudaGetLastError();
  return ICIKT_OK;
}

void icikt_plan_destroy(icikt_plan* p) { delete p; }

// The pipelined one-shot call on a staged plan (build_stage_table): uploads on the copy stream chunk by chunk,
// K1 of a chunk and the pair launches that need nothing beyond it on the compute stream, the results of
// a finished row block back on the copy stream while the next block runs.  `download` false: the results
// stay on the device (matrix output follows).  Same results as upload + columns + pairs + download: only
// the order in which the pairs are computed differs.
static int run_staged(icikt_plan* p, const ColumnSource& s, const double* global_na, int32_t n_global_na,
                      bool download, double* raw, double* pvalue, double* taumax, double* completeness,
                      int32_t* status, int64_t* counts, double* max_taumax) {
  if (!p || !p->staged) return fail(ICIKT_ERR_BAD_ARG, "not a staged plan");
  if (!s.csc() && (!s.data || s.ld < p->n)) return fail(ICIKT_ERR_BAD_ARG, "bad upload arguments");
  if (counts && !p->d_counts) return fail(ICIKT_ERR_BAD_ARG, "plan was created without want_counts");
  CK(cudaSetDevice(p->device));
  CK(p->d_data_own.reserve((size_t)p->n * p->C));
  p->d_data = p->d_data_own.get();
  p->ld = p->n;
  p->columns_done = false;
  p->pairs_done = false;
  p->staged_run = true;
  CK(cudaEventRecord(p->ev[0], p->stream));
  CK(cudaStreamWaitEvent(p->copy_stream, p->ev[0], 0));
  CK(cudaMemsetAsync(p->d_maxbits, 0, sizeof(unsigned long long), p->stream));
  int pair_launches = 0;
  const size_t L = p->stages.size();
  for (size_t l = 0; l < L; ++l) {
    const StageLaunch& st = p->stages[l];
    const Event* te = &p->time_ev[5 * l];
    if (st.col_hi > st.col_lo) {
      int rc = copy_columns_in(p, s, st.col_lo, st.col_hi, p->copy_stream);
      if (rc != ICIKT_OK) return rc;
      CK(cudaEventRecord(p->sync_ev[2 * l], p->copy_stream));
      if (st.col_hi == p->C) CK(cudaEventRecord(p->ev[1], p->copy_stream));
      CK(cudaStreamWaitEvent(p->stream, p->sync_ev[2 * l], 0));
      rc = plan_columns_impl(p, global_na, n_global_na, st.col_lo, st.col_hi, st.col_hi == p->C, st.col_lo == 0, te[0], te[1]);
      if (rc != ICIKT_OK) return rc;
    }
    const int rc = launch_pair_group(p, p->d_units.get(), st.unit_lo, st.unit_hi, st.max_unit_pairs, te[2], te[3], te[4], &pair_launches);
    if (rc != ICIKT_OK) return rc;
    CK(cudaEventRecord(p->sync_ev[2 * l + 1], p->stream));
  }
  p->tm.n_launches = (p->tm.n_launches & 0xffff) | (pair_launches << 16);
  p->pairs_done = true;
  bool d2h_started = false;  // ev[6]: the first result copy may start
  unsigned long long bits = 0;
  if (download) {
    const size_t np = (size_t)p->P, npad = std::max<size_t>(np, 1);
    struct Out { void* host; const unsigned char* dev; size_t elem; size_t res_off; };
    const Out outs[6] = {
        {raw, reinterpret_cast<const unsigned char*>(p->d_tau), sizeof(double), 0},
        {pvalue, reinterpret_cast<const unsigned char*>(p->d_p), sizeof(double), npad * sizeof(double)},
        {taumax, reinterpret_cast<const unsigned char*>(p->d_tm), sizeof(double), 2 * npad * sizeof(double)},
        {completeness, reinterpret_cast<const unsigned char*>(p->d_comp), sizeof(double), 3 * npad * sizeof(double)},
        {status, reinterpret_cast<const unsigned char*>(p->d_status), sizeof(int32_t),
         4 * npad * sizeof(double) + sizeof(unsigned long long)},
        {counts, reinterpret_cast<const unsigned char*>(p->d_counts.get()), sizeof(int64_t) * ICIKT_NCOUNTS, 0},
    };
    if (p->h_res) {
      // every block's copies into the pinned mirror are enqueued at once (each waits for its block), the
      // host then follows block by block and moves the ranges into the caller's arrays
      for (size_t l = 0; l < L; ++l) {
        const StageLaunch& st = p->stages[l];
        if (st.slot_hi <= st.slot_lo) continue;
        CK(cudaStreamWaitEvent(p->copy_stream, p->sync_ev[2 * l + 1], 0));
        if (!d2h_started) CK(cudaEventRecord(p->ev[6], p->copy_stream));
        d2h_started = true;
        for (int k = 0; k < 6; ++k) {
          if (!outs[k].host) continue;
          const size_t o = (size_t)st.slot_lo * outs[k].elem, b = (size_t)(st.slot_hi - st.slot_lo) * outs[k].elem;
          void* dst = (k == 5) ? static_cast<void*>(static_cast<unsigned char*>(outs[k].host) + o)
                               : static_cast<void*>(p->h_res.get() + outs[k].res_off + o);
          CK(cudaMemcpyAsync(dst, outs[k].dev + o, b, cudaMemcpyDeviceToHost, p->copy_stream));
        }
        CK(cudaEventRecord(p->sync_ev[2 * l], p->copy_stream));  // free since the block's columns were waited for
      }
      for (size_t l = 0; l < L; ++l) {
        const StageLaunch& st = p->stages[l];
        if (st.slot_hi <= st.slot_lo) continue;
        CK(cudaEventSynchronize(p->sync_ev[2 * l]));
        for (int k = 0; k < 5; ++k) {
          if (!outs[k].host) continue;
          const size_t o = (size_t)st.slot_lo * outs[k].elem, b = (size_t)(st.slot_hi - st.slot_lo) * outs[k].elem;
          host_copy(static_cast<unsigned char*>(outs[k].host) + o, p->h_res.get() + outs[k].res_off + o, b);
        }
      }
    } else {
      for (size_t l = 0; l < L; ++l) {
        const StageLaunch& st = p->stages[l];
        if (st.slot_hi <= st.slot_lo) continue;
        CK(cudaStreamWaitEvent(p->copy_stream, p->sync_ev[2 * l + 1], 0));
        if (!d2h_started) CK(cudaEventRecord(p->ev[6], p->copy_stream));
        d2h_started = true;
        for (int k = 0; k < 6; ++k) {
          if (!outs[k].host) continue;
          const size_t o = (size_t)st.slot_lo * outs[k].elem, b = (size_t)(st.slot_hi - st.slot_lo) * outs[k].elem;
          const int rc = staged_copy_out(p, static_cast<unsigned char*>(outs[k].host) + o, outs[k].dev + o, b, p->copy_stream);
          if (rc != ICIKT_OK) return rc;
        }
      }
    }
  }
  CK(cudaStreamWaitEvent(p->copy_stream, p->sync_ev[2 * L - 1], 0));
  if (!d2h_started) CK(cudaEventRecord(p->ev[6], p->copy_stream));
  CK(cudaMemcpyAsync(&bits, p->d_maxbits, sizeof(bits), cudaMemcpyDeviceToHost, p->copy_stream));
  CK(cudaEventRecord(p->ev[7], p->copy_stream));
  CK(cudaStreamSynchronize(p->copy_stream));
  CK(cudaStreamSynchronize(p->stream));
  if (max_taumax) {
    double v;
    std::memcpy(&v, &bits, sizeof(v));
    *max_taumax = bits ? v : std::nan("");
  }
  return ICIKT_OK;
}

// all pairs of a matrix this large go through the pipelined call (ICIKT_PIPELINE_MIN_BYTES, default 32 MB of
// input; ICIKT_NO_PIPELINE=1 switches it off)
static bool want_staged(int64_t n, int64_t C, const icikt_opts& o) {
  if (o.kernel != ICIKT_KERNEL_TILED || std::getenv("ICIKT_NO_PIPELINE")) return false;
  const size_t min_bytes = env_bytes("ICIKT_PIPELINE_MIN_BYTES", 32u << 20);
  return C >= 128 && sizeof(double) * (size_t)n * (size_t)C >= min_bytes;
}

// The cached plans: the per-pair and matrix calls' (one worker: g_cached, worker k of several: g_cached_multi[k]) and
// the windowed calls' (g_cached_edges, g_cached_wmulti[k]; their pair buffers hold one window).
static icikt_plan* g_cached = nullptr;
static icikt_plan* g_cached_multi[64] = {};
static icikt_plan* g_cached_edges = nullptr;
static icikt_plan* g_cached_wmulti[kMaxMatrixDevices] = {};
static std::mutex g_cache_mu;

// The plan of a call, cached in `slot` (the caller holds g_cache_mu): the slot's plan if n, C, `staged` and the
// options that shape a plan match (device, kernel, diagonal, pair range, counts, the complete-observations buffer),
// with the call's other options; otherwise a new plan takes the slot.
static int cached_plan(icikt_plan*& slot, int64_t n, int64_t C, const icikt_opts& o, bool staged, icikt_plan** out) {
  icikt_plan* p = slot;
  if (p && p->staged == staged && p->n == n && p->C == C && p->opts.device == o.device && p->opts.kernel == o.kernel &&
      p->opts.include_diag == o.include_diag && p->opts.pair_lo == o.pair_lo && p->opts.pair_hi == o.pair_hi &&
      p->want_counts == (o.want_counts != 0) && (o.perspective != ICIKT_PERSPECTIVE_COMPLETE || p->d_pw)) {
    p->opts.perspective = o.perspective;
    p->opts.alternative = o.alternative;
    p->opts.continuity = o.continuity;
    p->opts.na_inf = o.na_inf;
  } else {
    icikt_plan_destroy(p);
    slot = nullptr;
    const int rc = plan_create_impl(&p, n, C, nullptr, nullptr, 0, &o, staged);
    *out = p;
    if (rc != ICIKT_OK) return rc;
    slot = p;
  }
  *out = p;
  return ICIKT_OK;
}

int icikt_pair_from_index(int64_t C, int32_t include_diag, int64_t index, int32_t* i, int32_t* j) {
  if (C < 1 || !i || !j || index < 0) return fail(ICIKT_ERR_BAD_ARG, "bad pair index arguments");
  const int64_t ptri = tri_pairs(C);
  if (index >= ptri) {
    if (!include_diag || index >= ptri + C) return fail(ICIKT_ERR_BAD_ARG, "pair index out of range");
    *i = *j = (int32_t)(index - ptri);
    return ICIKT_OK;
  }
  // row r starts at r(2C-r-1)/2: invert with a float guess, then fix up exactly
  const double b = 2.0 * (double)C - 1.0;
  int64_t r = (int64_t)((b - std::sqrt(b * b - 8.0 * (double)index)) / 2.0);
  r = std::max<int64_t>(0, std::min<int64_t>(r, C - 2));
  while (r > 0 && row_start(r, C) > index) --r;
  while (r + 1 < C - 1 && row_start(r + 1, C) <= index) ++r;
  *i = (int32_t)r;
  *j = (int32_t)(r + 1 + (index - row_start(r, C)));
  return ICIKT_OK;
}

void icikt_release_workspace(void) {
  std::lock_guard<std::mutex> lock(g_cache_mu);
  if (g_cached) { icikt_plan_destroy(g_cached); g_cached = nullptr; }
  if (g_cached_edges) { icikt_plan_destroy(g_cached_edges); g_cached_edges = nullptr; }
  for (icikt_plan*& s : g_cached_multi)
    if (s) { icikt_plan_destroy(s); s = nullptr; }
  for (icikt_plan*& s : g_cached_wmulti)
    if (s) { icikt_plan_destroy(s); s = nullptr; }
}

int64_t icikt_stage_table(int64_t C, int32_t include_diag, int32_t cta_slots, int32_t n_blocks, int64_t cap_units,
                          int64_t* units, int64_t cap_launches, int64_t* launches, int64_t* n_launches) {
  if (C < 1 || cta_slots < 1 || n_blocks < 1) return fail(ICIKT_ERR_BAD_ARG, "bad stage table arguments");
  std::vector<PairUnit> U;
  std::vector<StageLaunch> S;
  build_stage_table(C, include_diag != 0, cta_slots, n_blocks, U, S);
  for (size_t k = 0; units && k < U.size() && (int64_t)k < cap_units; ++k) {
    units[4 * k + 0] = U[k].slot0;
    units[4 * k + 1] = U[k].col;
    units[4 * k + 2] = U[k].j0;
    units[4 * k + 3] = U[k].count;
  }
  for (size_t l = 0; launches && l < S.size() && (int64_t)l < cap_launches; ++l) {
    const int64_t row[6] = {S[l].col_lo, S[l].col_hi, S[l].unit_lo, S[l].unit_hi, S[l].slot_lo, S[l].slot_hi};
    std::memcpy(launches + 6 * l, row, sizeof(row));
  }
  if (n_launches) *n_launches = (int64_t)S.size();
  return (int64_t)U.size();
}

int icikt_launch_shape(int64_t n, int32_t tier, int32_t n_sm, int32_t complete_obs, int32_t* out) {
  if (n < 1 || n > tiled_max_n() || tier < 0 || tier > 2 || n_sm < 1 || !out)
    return fail(ICIKT_ERR_BAD_ARG, "bad launch shape arguments");
  const int64_t nwords = ((n + 31) & ~31LL) / 32, wstride = (nwords + 3) & ~3LL;
  const TiledShape sh = tiled_shape(n, tier, wstride, n_sm, 0, complete_obs == 0);
  const int cap = sh.warps * sh.kk * 256;
  out[0] = sh.warps;
  out[1] = sh.kk;
  out[2] = sh.region_bytes;
  out[3] = sh.inplace_kk != 0 ? 1 : (sh.gmem ? 2 : 0);
  out[4] = cap;
  // in place: rows of the other column's rank table one staging part holds (the counter area behind the sequence)
  out[5] = sh.inplace_kk != 0 ? (int)std::min<int64_t>((n + 63) & ~63LL, ((sh.region_bytes - 2 * cap) >> 1) & ~63) : 0;
  out[6] = sh.radix ? 1 : 0;
  return ICIKT_OK;
}

int icikt_measure_smem_bandwidth(int32_t device, double* g32, double* g128) {
  int rc = select_device(device);
  if (rc != ICIKT_OK) return rc;
  double a = 0, b = 0;
  if (measure_smem_bandwidth(&a, &b) < 0) return launch_fail("smem bandwidth kernel");
  if (g32) *g32 = a;
  if (g128) *g128 = b;
  return ICIKT_OK;
}

int icikt_measure_issue_rate(int32_t device, double* alu, double* fma, double* mixed) {
  int rc = select_device(device);
  if (rc != ICIKT_OK) return rc;
  double a = 0, f = 0, m = 0;
  if (measure_issue_rate(&a, &f, &m) < 0) return launch_fail("issue-rate kernel");
  if (alu) *alu = a;
  if (fma) *fma = f;
  if (mixed) *mixed = m;
  return ICIKT_OK;
}

}  // extern "C"

// ---- all pairs, filtered on the device (icikt_all_pairs_edges) ------------------------------------------------

struct icikt_edges {
  std::vector<EdgeRow> rows;
  std::vector<double> cor;
  int32_t j_offset = 0;  // a cross call's Cx: rows hold j as the matrix column of [X | Y], icikt_edges_copy gives Y's
  std::vector<double> padj;  // the _padj calls: the adjusted p-value of every row
  int64_t n_tests = -1;      // ... and m, the non-NaN p-values of the family; -1 without adjustment
};

// Pairs per window of the filtered calls, edges, top-k and cross (ICIKT_EDGE_WINDOW, at most 2^30).  The default 2^26
// keeps the window's buffers near 10 GB: the plan's pair buffers (68 B per pair) and the edge call's two
// selected-row buffers (40 B each), the top-k call's candidates (16 B) or the cross per-pair call's two result
// buffers (36 B each).
static int64_t edge_window() {
  const char* e = std::getenv("ICIKT_EDGE_WINDOW");
  const long long v = e ? std::atoll(e) : 0;
  return v > 0 ? std::min<long long>(v, 1LL << 30) : (1LL << 26);
}

static double max_of_bits(unsigned long long bits) {
  double v;
  std::memcpy(&v, &bits, sizeof(v));
  return bits ? v : std::nan("");
}

// The argument checks the filtered calls share, on the host before any device is touched.
static int check_window_args(const ColumnSource& s, int64_t n, int64_t C, const double* global_na,
                             int32_t n_global_na, const icikt_opts& o) {
  if (n < 1 || C < 1) return fail(ICIKT_ERR_BAD_ARG, "n and C must be >= 1");
  if (!s.csc() && (!s.data || s.ld < n)) return fail(ICIKT_ERR_BAD_ARG, "data must not be NULL and ld >= n");
  if (n > tiled_max_n()) return fail(ICIKT_ERR_TOO_LONG, "n exceeds icikt_max_n()");
  if (C > 2147483647LL) return fail(ICIKT_ERR_BAD_ARG, "too many columns");
  if (n_global_na < 0 || (n_global_na > 0 && !global_na)) return fail(ICIKT_ERR_BAD_ARG, "bad global_na");
  if (o.pair_lo != 0 || o.pair_hi != 0)
    return fail(ICIKT_ERR_BAD_ARG, "the filtered call covers all pairs: pair_lo and pair_hi must be 0");
  if (o.perspective != ICIKT_PERSPECTIVE_GLOBAL && o.perspective != ICIKT_PERSPECTIVE_LOCAL)
    return fail(ICIKT_ERR_BAD_ARG, "the filtered call takes the global or the local perspective");
  if (o.kernel != ICIKT_KERNEL_TILED) return fail(ICIKT_ERR_BAD_ARG, "the filtered call needs the tiled kernel");
  if (o.want_counts) return fail(ICIKT_ERR_BAD_ARG, "the filtered call returns no counts (want_counts)");
  return ICIKT_OK;
}

// the filter and the result pointer of the edge calls
static int check_filter_args(const icikt_edge_filter* f, icikt_edges** out) {
  if (!out) return fail(ICIKT_ERR_BAD_ARG, "out is NULL");
  *out = nullptr;
  if (!f) return fail(ICIKT_ERR_BAD_ARG, "filter is NULL");
  if (f->max_edges < 0) return fail(ICIKT_ERR_BAD_ARG, "max_edges must be >= 0 (0: no limit)");
  return ICIKT_OK;
}

static int check_edge_args(const ColumnSource& s, int64_t n, int64_t C, const double* global_na, int32_t n_global_na,
                           const icikt_opts& o, const icikt_edge_filter* f, icikt_edges** out) {
  const int rc = check_filter_args(f, out);
  return rc == ICIKT_OK ? check_window_args(s, n, C, global_na, n_global_na, o) : rc;
}

// k and by of the top-k calls
static int check_k_by(int32_t k, int32_t by) {
  if (k < 1 || k > ICIKT_TOPK_MAX) return fail(ICIKT_ERR_BAD_ARG, "k must be in [1, ICIKT_TOPK_MAX]");
  if (by != ICIKT_TOPK_ABS && by != ICIKT_TOPK_SIGNED)
    return fail(ICIKT_ERR_BAD_ARG, "by must be ICIKT_TOPK_ABS or ICIKT_TOPK_SIGNED");
  return ICIKT_OK;
}

static int check_topk_args(const ColumnSource& s, int64_t n, int64_t C, const double* global_na, int32_t n_global_na,
                           const icikt_opts& o, int32_t k, int32_t by, const int32_t* index) {
  const int rc = check_k_by(k, by);
  if (rc != ICIKT_OK) return rc;
  if (!index) return fail(ICIKT_ERR_BAD_ARG, "index is NULL");
  if (o.include_diag) return fail(ICIKT_ERR_BAD_ARG, "the top-k call ranks partners d != c: include_diag must be 0");
  return check_window_args(s, n, C, global_na, n_global_na, o);
}


// the window walk's events, readbacks and staging chunks (kept with the plan)
static int ensure_walk_buffers(icikt_plan* p) {
  if (!p->copy_stream) ECK(p->copy_stream.create());
  for (auto& evs : p->eev)
    for (Event& e : evs)
      if (!e) ECK(e.create());
  ECK(p->h_estat.reserve(4));
  ECK(p->d_etotal.reserve(2));
  return ensure_stage(p);
}

// the edge selection's buffers for windows of W pairs (kept with the plan)
static int ensure_edge_buffers(icikt_plan* p, int64_t W) {
  const int rc = ensure_walk_buffers(p);
  if (rc != ICIKT_OK) return rc;
  const int64_t tiles = (W + kEdgeTile - 1) / kEdgeTile;
  ECK(p->d_emask.reserve((size_t)tiles * (kEdgeTile / 32)));
  ECK(p->d_etile.reserve((size_t)tiles));
  for (auto& rows : p->d_erows) ECK(rows.reserve((size_t)W));
  return ICIKT_OK;
}

// the top-k selection's buffers: candidates of a window of W pairs, and lists of k entries for L columns (C, or the
// requested sides of a cross call)
static int ensure_topk_buffers(icikt_plan* p, int64_t W, int k, int64_t L) {
  const int rc = ensure_walk_buffers(p);
  if (rc != ICIKT_OK) return rc;
  ECK(p->d_tcand.reserve(2 * (size_t)W));
  ECK(p->d_tcount.reserve((size_t)L));
  ECK(p->d_tcol.reserve((size_t)L));
  ECK(p->d_tidx.reserve((size_t)(L * k)));
  ECK(p->d_tlist.reserve(4 * (size_t)(L * k)));
  return ICIKT_OK;
}

// the merged lists of a block of columns (top-k over several devices): `entries` = columns of the block x k
static int ensure_merge_buffers(icikt_plan* p, size_t entries) {
  ECK(p->d_mn.reserve((size_t)p->C));
  ECK(p->d_midx.reserve(entries));
  ECK(p->d_mlist.reserve(4 * entries));
  return ensure_stage(p);
}

// room for `need` units in both window unit buffers (device and pinned host)
static int ensure_window_units(icikt_plan* p, size_t need) {
  size_t have = p->d_wunits[0].size();
  for (int b = 0; b < 2; ++b) have = std::min({have, p->d_wunits[b].size(), p->h_wunits[b].size()});
  if (need <= have) return ICIKT_OK;
  CK(cudaStreamSynchronize(p->stream));  // the other buffer may still be read by the previous window
  const size_t cap = std::max(need + need / 4, 2 * have);
  for (int b = 0; b < 2; ++b) {
    ECK(p->d_wunits[b].reserve(cap));
    ECK(p->h_wunits[b].reserve(cap));
  }
  return ICIKT_OK;
}

// what the window walk adds up: event times, launches, and the maximum taumax so far (bits)
struct WalkTotals {
  float up_ms = 0.f, pairs_ms = 0.f, epi_ms = 0.f;
  int launches = 0;
  unsigned long long bits = 0;
};

// The upload of columns [c_lo, c_hi) of [X | Y] (y: Y of a cross call, from column s.C on, or null): X's part, then
// Y's part.  X's CSC arrays occupy the plan's CSC buffers, which Y's overwrite (and may reallocate), so X's part is
// expanded before Y's is uploaded; x_launches: that expansion's launches.
static int upload_span(icikt_plan* p, const ColumnSource& s, const ColumnSource* y, int64_t c_lo, int64_t c_hi,
                       int* x_launches) {
  *x_launches = 0;
  int rc = upload_columns(p, s, std::min(c_lo, s.C), std::min(c_hi, s.C));
  if (rc != ICIKT_OK || !y || c_hi <= s.C) return rc;
  *x_launches = expand_columns(p);
  if (*x_launches < 0) return ICIKT_ERR_CUDA;
  if (*x_launches > 0 && y->csc()) CK(cudaStreamSynchronize(p->stream));
  rc = copy_columns_in(p, *y, std::max<int64_t>(c_lo - s.C, 0), c_hi - s.C, p->stream, s.C);
  if (rc != ICIKT_OK) return rc;
  CK(cudaEventRecord(p->ev[1], p->stream));
  return ICIKT_OK;
}

// upload and K1 of all columns on one device (the column phase of a multi-device job without peer gather).  A cross
// job passes Y as `y`: its columns land behind X's, and K1 runs once over all columns of [X | Y].
static int window_columns(icikt_plan* p, const ColumnSource& s, const double* global_na, int32_t n_global_na,
                          const ColumnSource* y = nullptr) {
  int x_launches = 0;
  int rc = upload_span(p, s, y, 0, p->C, &x_launches);
  if (rc == ICIKT_OK) rc = plan_columns_impl(p, global_na, n_global_na, 0, p->C, true);
  p->tm.n_launches += x_launches;
  return rc;
}

// The unit builders of the two pair orders the window walk knows, for pairs [lo, hi) with slots from lo.
// combn order (all-pairs calls; the diagonal follows if include_diag):
static auto combn_order(const icikt_plan* p) {
  return [C = p->C, diag = p->opts.include_diag != 0](int64_t lo, int64_t hi, int64_t slots, std::vector<PairUnit>& U) {
    int32_t row = 0, col = 0;
    if (lo < tri_pairs(C)) icikt_pair_from_index(C, 0, lo, &row, &col);
    range_units(C, diag, lo, hi, slots, U, row);
  };
}
// cross order of Cx x Cy (icikt_cross.cuh):
static auto cross_order(int64_t Cx, int64_t Cy) {
  return [Cx, Cy](int64_t lo, int64_t hi, int64_t slots, std::vector<PairUnit>& U) { cross_units(Cx, Cy, lo, hi, slots, U); };
}

// The window walk of the filtered calls, on a plan whose pair buffers hold W pairs and whose columns are prepared
// (K1 enqueued): pairs [first, last) of a pair order in windows of W; order(lo, hi, slots, U) appends the units of
// pairs [lo, hi) (combn_order or cross_order).  Window w is enqueued (units, K2, K3,
// `select`, the readback of the maximum so far) before the host waits for window w - 1 and runs `collect` for it;
// d_maxbits is not reset between windows, so K3's atomicMax leaves that maximum.  select(w, b, units, n_units,
// n_slots) enqueues the selection of window w on p->stream (b: its buffer, 0 or 1); collect(w, b) runs once that
// has completed.
template <class Order, class Select, class Collect>
static int walk_windows(icikt_plan* p, const Order& order, int64_t first, int64_t last, int64_t W, WalkTotals& tot,
                        Select&& select, Collect&& collect) {
  tot.launches = p->tm.n_launches;
  CK(cudaMemsetAsync(p->d_maxbits, 0, sizeof(unsigned long long), p->stream));
  const int64_t nwin = (last - first + W - 1) / W, slots = (int64_t)p->n_sm * 2;
  std::vector<PairUnit> U;
  int rc = ICIKT_OK;

  auto enqueue = [&](int64_t w) -> int {
    const int b = (int)(w & 1);
    const int64_t lo = first + w * W, hi = std::min(last, lo + W);
    U.clear();
    order(lo, hi, slots, U);
    int r = ensure_window_units(p, U.size());
    if (r != ICIKT_OK) return r;
    // the buffer was last read by window w - 2, whose selection the host has waited for
    std::memcpy(p->h_wunits[b].get(), U.data(), sizeof(PairUnit) * U.size());
    int max_unit = 1;
    for (const PairUnit& u : U) max_unit = std::max(max_unit, (int)u.count);
    const Event* e = p->eev[b];
    CK(cudaEventRecord(e[0], p->stream));
    CK(cudaMemcpyAsync(p->d_wunits[b].get(), p->h_wunits[b].get(), sizeof(PairUnit) * U.size(), cudaMemcpyHostToDevice, p->stream));
    CK(cudaEventRecord(e[1], p->stream));
    r = launch_pair_group(p, p->d_wunits[b].get(), 0, (int64_t)U.size(), max_unit, e[2], e[3], e[4], &tot.launches);
    if (r != ICIKT_OK) return r;
    r = select(w, b, p->d_wunits[b].get(), (int64_t)U.size(), hi - lo);
    if (r != ICIKT_OK) return r;
    CK(cudaMemcpyAsync(p->h_estat.get() + 2 * b + 1, p->d_maxbits, sizeof(unsigned long long), cudaMemcpyDeviceToHost, p->stream));
    CK(cudaEventRecord(e[5], p->stream));
    return ICIKT_OK;
  };

  auto wait = [&](int64_t w) -> int {
    const int b = (int)(w & 1);
    const Event* e = p->eev[b];
    CK(cudaEventSynchronize(e[5]));
    tot.bits = p->h_estat.get()[2 * b + 1];
    tot.up_ms += ev_ms(e[0], e[1]);
    tot.pairs_ms += ev_ms(e[2], e[3]);
    tot.epi_ms += ev_ms(e[3], e[5]);
    return collect(w, b);
  };

  for (int64_t w = 0; w <= nwin; ++w) {
    if (w < nwin && (rc = enqueue(w)) != ICIKT_OK) return rc;
    if (w > 0 && (rc = wait(w - 1)) != ICIKT_OK) return rc;
  }
  return ICIKT_OK;
}

// the end of a walk: both streams drained, then the timings (d2h_ms: the caller's copies out)
static int finish_walk(icikt_plan* p, const WalkTotals& tot, float d2h_ms, icikt_timings* timings) {
  CK(cudaEventRecord(p->ev[4], p->copy_stream));
  CK(cudaStreamWaitEvent(p->stream, p->ev[4], 0));
  CK(cudaEventRecord(p->ev[5], p->stream));
  CK(cudaEventSynchronize(p->ev[5]));
  if (timings) {
    std::memset(timings, 0, sizeof(*timings));
    timings->h2d_ms = ev_ms(p->ev[0], p->ev[1]) + tot.up_ms;
    timings->columns_ms = ev_ms(p->ev[2], p->ev[3]);
    timings->pairs_ms = tot.pairs_ms;
    timings->epilogue_ms = tot.epi_ms;
    timings->d2h_ms = d2h_ms;
    timings->total_ms = ev_ms(p->ev[0], p->ev[5]);
    timings->n_launches = tot.launches;
    cudaGetLastError();
  }
  return ICIKT_OK;
}

// ---- adjusted p-values (the _padj edge calls): every walker keeps the count of the non-NaN p-values of its slice and
// the keys of its candidates, the p-values <= the candidate bound (icikt_padj.cuh: a prefix of the ascending order
// that holds every row whose adjusted value can pass).  The buffer grows geometrically; it always has room for the two
// windows whose counts the host has not read back yet.
struct PadjPart {
  int device = -1;                           // where the buffers live (-1: not set up)
  DeviceArray<unsigned long long> d_cnt;     // [2]: non-NaN p-values, candidates
  PinnedArray<unsigned long long> h_cnt;     // [2][2]: the readback of d_cnt, per window buffer
  DeviceArray<unsigned long long> d_keys;    // its size is the capacity
  int64_t known = 0;                         // candidates as of the last readback
  int64_t m = 0, K = 0;                      // after the walk: non-NaN p-values and candidates
  double bound = 0.0;                        // the candidate bound (NaN: every non-NaN p-value)
  ~PadjPart() {
    if (device >= 0) cudaSetDevice(device);
  }
};

// room in a's buffer for `more` candidates beyond those last read back (set up on p's device at the first window)
static int padj_room(icikt_plan* p, PadjPart& a, int64_t more) {
  if (a.device < 0) {
    a.device = p->device;
    ECK(a.d_cnt.reserve(2));
    ECK(a.h_cnt.reserve(4));
    std::memset(a.h_cnt.get(), 0, 4 * sizeof(unsigned long long));
    CK(cudaMemsetAsync(a.d_cnt.get(), 0, 2 * sizeof(unsigned long long), p->stream));
  }
  if (a.known + more <= (int64_t)a.d_keys.size()) return ICIKT_OK;
  CK(cudaStreamSynchronize(p->stream));  // the windows in flight append to the old buffer
  unsigned long long now[2];
  CK(cudaMemcpy(now, a.d_cnt.get(), sizeof(now), cudaMemcpyDeviceToHost));
  a.known = (int64_t)now[1];
  const int64_t cap = std::max(2 * (int64_t)a.d_keys.size(), a.known + more);
  DeviceArray<unsigned long long> keys;
  if (keys.reserve((size_t)cap) != cudaSuccess) {
    cudaGetLastError();
    return fail(ICIKT_ERR_ALLOC, "device allocation for " + std::to_string(cap) + " p-value candidates failed (" +
                                     std::to_string(a.known) + " held)");
  }
  if (a.known) {
    const cudaError_t e = cudaMemcpy(keys.get(), a.d_keys.get(), sizeof(unsigned long long) * (size_t)a.known,
                                     cudaMemcpyDeviceToDevice);
    if (e != cudaSuccess) return cuda_fail(e, "p-value candidates");
  }
  a.d_keys = std::move(keys);
  return ICIKT_OK;
}

// The rows all walkers of one filtered call hold, for max_edges: one walker on one device, one per device in the
// multi-device call.  A walker that takes the sum over the limit raises `stop`, and the others fail at their next
// window boundary.
struct EdgeHeld {
  std::atomic<int64_t> total{0};
  std::atomic<bool> stop{false};
};

static int edge_limit_fail(const icikt_edge_filter& f, int64_t held, const std::string& where) {
  return fail(ICIKT_ERR_LIMIT, "more than max_edges = " + std::to_string(f.max_edges) + " pairs pass the filter (" +
                                   std::to_string(held) + where + ")");
}

// The filtered call's walk over pairs [first, last): per window, the edge selection and the readback of its row
// count; once the host has waited for a window, its rows are copied out on the copy stream and appended to `rows`,
// and the rows held are re-trimmed against the new maximum (this walk's own: at most the final one, so the rows
// stay a superset of the final edges).  The plan's edge buffers hold windows of W pairs.
template <class Order>
static int edge_walk(icikt_plan* p, const Order& order, const icikt_edge_filter& f, int64_t first, int64_t last,
                     int64_t W, std::vector<EdgeRow>& rows, EdgeHeld& held, WalkTotals& tot, float& d2h_ms,
                     PadjPart* adj = nullptr) {
  const double t = f.min_abs_cor;
  const bool scale = f.scale_max != 0;
  const bool retrim = scale && t == t;
  const int64_t nwin = (last - first + W - 1) / W;
  unsigned long long trimmed_bits = 0;

  auto select = [&](int64_t, int b, const PairUnit* units, int64_t n_units, int64_t n_slots) -> int {
    EdgeSelect es;
    es.units = units;
    es.n_units = n_units;
    es.n_slots = n_slots;
    es.tau = p->d_tau;
    es.pvalue = p->d_p;
    es.taumax = p->d_tm;
    es.completeness = p->d_comp;
    es.status = p->d_status;
    es.max_taumax_bits = p->d_maxbits;
    es.min_abs_cor = f.min_abs_cor;
    es.max_pvalue = f.max_pvalue;
    es.scale_max = scale ? 1 : 0;
    es.mask = p->d_emask.get();
    es.tile_offset = p->d_etile.get();
    es.total = p->d_etotal.get() + b;
    es.rows = p->d_erows[b].get();
    const int l = launch_edge_select(es, p->stream);
    if (l < 0) return launch_fail("edge selection kernels");
    tot.launches += l;
    CK(cudaMemcpyAsync(p->h_estat.get() + 2 * b, p->d_etotal.get() + b, sizeof(unsigned long long), cudaMemcpyDeviceToHost, p->stream));
    if (adj) {  // the window's non-NaN count and candidates, in the epilogue's time
      const int r = padj_room(p, *adj, 2 * W);
      if (r != ICIKT_OK) return r;
      CK(padj_candidates(p->d_p, n_slots, adj->bound, adj->d_cnt.get(), adj->d_keys.get(), p->stream));
      CK(cudaMemcpyAsync(adj->h_cnt.get() + 2 * b, adj->d_cnt.get(), 2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, p->stream));
    }
    return ICIKT_OK;
  };

  auto collect = [&](int64_t w, int b) -> int {
    if (held.stop) return edge_limit_fail(f, held.total, " held when another device reached the limit");
    const unsigned long long cnt = p->h_estat.get()[2 * b];
    const unsigned long long bits = tot.bits;
    if (adj) adj->known = std::max<int64_t>(adj->known, (int64_t)adj->h_cnt.get()[2 * b + 1]);
    const size_t before = rows.size();
    if (cnt) {
      const size_t old = rows.size();
      try {
        rows.resize(old + (size_t)cnt);
      } catch (const std::bad_alloc&) {
        return fail(ICIKT_ERR_ALLOC, "out of host memory for the selected rows");
      }
      CK(cudaEventRecord(p->ev[6], p->copy_stream));
      const int r = staged_copy_out(p, rows.data() + old, p->d_erows[b].get(), sizeof(EdgeRow) * (size_t)cnt, p->copy_stream);
      if (r != ICIKT_OK) return r;
      CK(cudaEventRecord(p->ev[7], p->copy_stream));
      CK(cudaEventSynchronize(p->ev[7]));
      d2h_ms += ev_ms(p->ev[6], p->ev[7]);
    }
    if (retrim && bits != trimmed_bits) {  // the maximum grew: rows held from earlier windows may no longer pass
      const double m = max_of_bits(bits);
      rows.erase(std::remove_if(rows.begin(), rows.end(), [&](const EdgeRow& r) { return !edge_prefilter(r.raw, t, m); }),
                 rows.end());
      trimmed_bits = bits;
    }
    const int64_t sum = held.total += (int64_t)rows.size() - (int64_t)before;
    if (f.max_edges > 0 && sum > f.max_edges) {
      held.stop = true;
      return edge_limit_fail(f, sum, " held after " + std::to_string(w + 1) + " of " + std::to_string(nwin) + " windows");
    }
    return ICIKT_OK;
  };

  const int rc = walk_windows(p, order, first, last, W, tot, select, collect);
  if (rc != ICIKT_OK || !adj || adj->device < 0) return rc;
  unsigned long long now[2];
  CK(cudaStreamSynchronize(p->stream));
  CK(cudaMemcpy(now, adj->d_cnt.get(), sizeof(now), cudaMemcpyDeviceToHost));
  adj->m = (int64_t)now[0];
  adj->K = (int64_t)now[1];
  return ICIKT_OK;
}

// The end of the filtered call, on one device or several: the rows held, in pair order, get the exact predicate with
// the final maximum M, then `adjust` (the _padj calls: adjusted p-values and their trim), the max_edges check and cor.
static int edge_result(icikt_edges* res, const icikt_edge_filter& f, double M,
                       const std::function<int(icikt_edges*)>& adjust = nullptr) {
  std::vector<EdgeRow>& rows = res->rows;
  const double t = f.min_abs_cor;
  const bool scale = f.scale_max != 0;
  if (scale && t == t)
    rows.erase(std::remove_if(rows.begin(), rows.end(), [&](const EdgeRow& r) { return !edge_keep_final(r.raw, t, true, M); }),
               rows.end());
  if (adjust) {
    const int rc = adjust(res);
    if (rc != ICIKT_OK) return rc;
  }
  if (f.max_edges > 0 && (int64_t)rows.size() > f.max_edges) return edge_limit_fail(f, (int64_t)rows.size(), "");
  try {
    res->cor.resize(rows.size());
  } catch (const std::bad_alloc&) {
    return fail(ICIKT_ERR_ALLOC, "out of host memory for cor");
  }
  for (size_t k = 0; k < rows.size(); ++k) res->cor[k] = scale ? rows[k].raw / M : rows[k].raw;
  return ICIKT_OK;
}

// The top-k call: per window, the top-k selection merges the window's candidates into the lists on the device;
// nothing comes back until the last window, then the lists are copied out once and cor is formed with the
// final maximum.
static_assert(kTopkMax == ICIKT_TOPK_MAX, "the merge kernel holds one list entry per thread");
struct TopkOut {
  int32_t *index, *n_neighbors;
  double *cor, *raw, *pvalue, *taumax, *completeness;
};

// The top-k call's walk over pairs [first, last) of `order`: the lists of columns [c_lo, c_hi) start empty and every
// window's candidates are merged into them on the device.  The plan's top-k buffers hold windows of W pairs and
// lists of k entries for those columns.
template <class Order>
static int topk_walk(icikt_plan* p, const Order& order, int64_t c_lo, int64_t c_hi, int k, int by, int64_t first,
                     int64_t last, int64_t W, WalkTotals& tot) {
  const int64_t ck = (c_hi - c_lo) * k;
  CK(cudaMemsetAsync(p->d_tcol.get(), 0, sizeof(TopkCol) * (size_t)(c_hi - c_lo), p->stream));
  auto select = [&](int64_t, int b, const PairUnit* units, int64_t n_units, int64_t n_slots) -> int {
    TopkSelect ts;
    ts.units = units;
    ts.n_units = n_units;
    ts.n_slots = n_slots;
    ts.tau = p->d_tau;
    ts.pvalue = p->d_p;
    ts.taumax = p->d_tm;
    ts.completeness = p->d_comp;
    ts.status = p->d_status;
    ts.c_lo = c_lo;
    ts.c_hi = c_hi;
    ts.k = k;
    ts.by = by;
    ts.col_count = p->d_tcount.get();
    ts.total = p->d_etotal.get() + b;
    ts.cand = p->d_tcand.get();
    ts.col = p->d_tcol.get();
    ts.idx = p->d_tidx.get();
    ts.raw = p->d_tlist.get();
    ts.pv = p->d_tlist.get() + ck;
    ts.tm = p->d_tlist.get() + 2 * ck;
    ts.comp = p->d_tlist.get() + 3 * ck;
    const int l = launch_topk_select(ts, p->stream);
    if (l < 0) return launch_fail("top-k selection kernels");
    tot.launches += l;
    return ICIKT_OK;
  };
  return walk_windows(p, order, first, last, W, tot, select, [](int64_t, int) { return ICIKT_OK; });
}

// raw for cor when the caller wants cor but not raw
static int topk_raw_buffer(const TopkOut& out, int64_t ck, std::vector<double>& own, double** raw) {
  *raw = out.raw;
  if (out.raw || !out.cor) return ICIKT_OK;
  try {
    own.resize((size_t)ck);
  } catch (const std::bad_alloc&) {
    return fail(ICIKT_ERR_ALLOC, "out of host memory for the lists");
  }
  *raw = own.data();
  return ICIKT_OK;
}

// The host's part of the top-k result once the lists of columns [0, C) are in the caller's arrays (raw: out.raw or
// the buffer topk_raw_buffer gave): n_neighbors from held(c), cor = raw / M (scale) or raw, and the padding.
template <class Held>
static void topk_fill_host(const TopkOut& out, int64_t C, int k, Held&& held, const double* raw, bool scale, double M) {
  const double qnan = std::nan("");
  for (int64_t c = 0; c < C; ++c) {
    const int64_t h = held(c), base = c * k;
    if (out.n_neighbors) out.n_neighbors[c] = (int32_t)h;
    if (out.cor)
      for (int64_t r = 0; r < h; ++r) out.cor[base + r] = scale ? raw[base + r] / M : raw[base + r];
    for (int64_t r = h; r < k; ++r) {
      out.index[base + r] = -1;
      for (double* a : {out.cor, out.raw, out.pvalue, out.taumax, out.completeness})
        if (a) a[base + r] = qnan;
    }
  }
}

// One side of a top-k result in the caller's arrays: rows [row0, row0 + cols) of the device lists.  `shift` is
// subtracted from its partners once they are copied (a cross call's x side: plan column Cx + j becomes Y's index j);
// raw: out.raw or the buffer topk_raw_buffer gave.
struct TopkSide {
  TopkOut out;
  int64_t row0, cols;
  int32_t shift;
  std::vector<double> raw_own;
  double* raw = nullptr;
};

// The host's part once every side's lists are in the caller's arrays: the partner shift, then topk_fill_host;
// held(row): the entries of list row `row`.
template <class Held>
static void topk_sides_finish(std::vector<TopkSide>& sides, int k, Held&& held, bool scale, double M) {
  for (TopkSide& sd : sides) {
    auto side_held = [&](int64_t c) { return (int64_t)held(sd.row0 + c); };
    if (sd.shift)
      for (int64_t c = 0; c < sd.cols; ++c)
        for (int64_t r = 0, h = side_held(c); r < h; ++r) sd.out.index[c * k + r] -= sd.shift;
    topk_fill_host(sd.out, sd.cols, k, side_held, sd.raw, scale, M);
  }
}

// ---- edge counts (icikt_all_pairs_count_edges, icikt_cross_count_edges): per window, the tally kernel adds the
// window's passing pairs to the plan's counters; nothing comes back until the last window.
static_assert(kCountFiltersMax == ICIKT_COUNT_FILTERS_MAX, "the tally kernel takes every filter in its parameters");
struct CountSpec {
  int T = 0;
  double t[kCountFiltersMax], a[kCountFiltersMax];  // min_abs_cor, max_pvalue of every filter (NaN: no condition)
  bool degree = false;                              // the caller wants degrees
  bool components = false;                          // the component calls: forests, hooks and labels
};

// one of the caller's degree tables: plan columns [c_lo, c_hi), entry (c - c_lo) * T + f (may be null)
struct DegreeOut {
  int64_t* out;
  int64_t c_lo, c_hi;
};

// one of the caller's label tables, in the layout of DegreeOut
struct ComponentOut {
  int32_t* out;
  int64_t c_lo, c_hi;
};

// The edge-count walk over pairs [first, last) of `order`: the counters start at zero and every window's tally adds
// to them; then they come back once into `out` (d_ecount's layout) and d2h_ms receives the time of that copy.  With
// cs.components the tally also unites each filter's forest, whose labels (the kernel that resolves them included in
// d2h_ms) come back into `labels`, [T][C] filter-major.  The forest is set to parent[v] = v just before the first
// window's tally, on the same stream, so that its time counts in epilogue_ms with the tally's.
template <class Order>
static int count_walk(icikt_plan* p, const Order& order, const CountSpec& cs, int64_t first, int64_t last, int64_t W,
                      WalkTotals& tot, std::vector<unsigned long long>& out, std::vector<int32_t>& labels,
                      float& d2h_ms) {
  const size_t hooks_at = 16 + (size_t)cs.T + (cs.degree ? (size_t)cs.T * (size_t)p->C : 0);
  const size_t entries = hooks_at + (cs.components ? (size_t)cs.T : 0);
  const size_t n_labels = cs.components ? (size_t)cs.T * (size_t)p->C : 0;
  ECK(p->d_ecount.reserve(entries));
  unsigned long long* c = p->d_ecount.get();
  CK(cudaMemsetAsync(c, 0, sizeof(unsigned long long) * entries, p->stream));
  if (cs.components) ECK(p->d_eparent.reserve(n_labels));
  auto select = [&](int64_t w, int, const PairUnit* units, int64_t n_units, int64_t n_slots) -> int {
    if (cs.components && w == 0) {
      const int l = launch_component_init(p->d_eparent.get(), cs.T, p->C, p->stream);
      if (l < 0) return launch_fail("component init kernel");
      tot.launches += l;
    }
    EdgeTally et;
    et.units = units;
    et.n_units = n_units;
    et.n_slots = n_slots;
    et.tau = p->d_tau;
    et.pvalue = p->d_p;
    et.status = p->d_status;
    et.n_filters = cs.T;
    et.C = p->C;
    std::memcpy(et.min_abs_cor, cs.t, sizeof(et.min_abs_cor));
    std::memcpy(et.max_pvalue, cs.a, sizeof(et.max_pvalue));
    et.status_counts = c;
    et.n_pass = c + 16;
    et.degree = cs.degree ? c + 16 + cs.T : nullptr;
    et.parent = cs.components ? p->d_eparent.get() : nullptr;
    et.hooks = cs.components ? c + hooks_at : nullptr;
    const int l = launch_edge_tally(et, p->stream);
    if (l < 0) return launch_fail("edge tally kernel");
    tot.launches += l;
    return ICIKT_OK;
  };
  int rc = walk_windows(p, order, first, last, W, tot, select, [](int64_t, int) { return ICIKT_OK; });
  if (rc != ICIKT_OK) return rc;
  try {
    out.resize(entries);
    labels.resize(n_labels);
  } catch (const std::bad_alloc&) {
    return fail(ICIKT_ERR_ALLOC, "out of host memory for the counters");
  }
  CK(cudaEventRecord(p->ev[6], p->stream));
  if (cs.components) {
    const int l = launch_component_labels(p->d_eparent.get(), cs.T, p->C, p->stream);
    if (l < 0) return launch_fail("component labels kernel");
    tot.launches += l;
  }
  rc = staged_copy_out(p, out.data(), c, sizeof(unsigned long long) * entries, p->stream);
  if (rc == ICIKT_OK && n_labels)
    rc = staged_copy_out(p, labels.data(), p->d_eparent.get(), sizeof(int32_t) * n_labels, p->stream);
  if (rc != ICIKT_OK) return rc;
  CK(cudaEventRecord(p->ev[7], p->stream));
  CK(cudaEventSynchronize(p->ev[7]));
  d2h_ms = ev_ms(p->ev[6], p->ev[7]);
  return ICIKT_OK;
}

extern "C" {

int64_t icikt_edges_count(const icikt_edges* e) { return e ? (int64_t)e->rows.size() : 0; }

int icikt_edges_copy(const icikt_edges* e, int32_t* i, int32_t* j, double* cor, double* raw, double* pvalue,
                     double* taumax, double* completeness) {
  if (!e) return fail(ICIKT_ERR_BAD_ARG, "edges is NULL");
  const size_t m = e->rows.size();
  for (size_t k = 0; k < m; ++k) {
    const EdgeRow& r = e->rows[k];
    if (i) i[k] = r.i;
    if (j) j[k] = r.j - e->j_offset;
    if (raw) raw[k] = r.raw;
    if (pvalue) pvalue[k] = r.pvalue;
    if (taumax) taumax[k] = r.taumax;
    if (completeness) completeness[k] = r.completeness;
  }
  if (cor && m) std::memcpy(cor, e->cor.data(), sizeof(double) * m);
  return ICIKT_OK;
}

void icikt_edges_free(icikt_edges* e) { delete e; }

}  // extern "C"

// ---- cross calls: every column of X against every column of Y (icikt_cross_pairs / _edges / _topk) ------------
// The plan holds [X | Y] (Y from column Cx on) and K1 runs once over all Cx + Cy columns; the window walk covers the
// cross order (icikt_cross.cuh), whose pair (i, j) is the plan's pair (i, Cx + j) staged with x column i.

// One matrix of a cross call, checked on the host: exactly one form, C >= 1, ld >= n or a valid CSC matrix.
static int cross_source(const icikt_input* in, const char* name, int64_t n, ColumnSource* out) {
  const std::string m = std::string("matrix ") + name + ": ";
  if (!in) return fail(ICIKT_ERR_BAD_ARG, m + "the input descriptor is NULL");
  if ((in->data != nullptr) == (in->colptr != nullptr))
    return fail(ICIKT_ERR_BAD_ARG, m + "set exactly one of data (dense) and colptr (CSC)");
  if (in->C < 1) return fail(ICIKT_ERR_BAD_ARG, m + "C must be >= 1");
  if (in->data) {
    if (in->ld < n) return fail(ICIKT_ERR_BAD_ARG, m + "ld must be >= n");
    *out = dense_source(in->data, in->ld, in->C);
    return ICIKT_OK;
  }
  const int rc = check_csc(in->colptr, in->rowidx, in->values, n, in->C);
  if (rc != ICIKT_OK) return fail(rc, m + g_err);
  *out = csc_source(in->colptr, in->rowidx, in->values, in->C);
  return ICIKT_OK;
}

// The argument checks all cross calls share, before any device is touched.  `ranged`: the call takes pair_lo /
// pair_hi (within [0, Cx Cy]); the others refuse them.
static int check_cross_args(const icikt_input* x, const icikt_input* y, int64_t n, const double* global_na,
                            int32_t n_global_na, const icikt_opts& o, bool ranged, ColumnSource* sx, ColumnSource* sy) {
  if (n < 1) return fail(ICIKT_ERR_BAD_ARG, "n must be >= 1");
  int rc = cross_source(x, "x", n, sx);
  if (rc == ICIKT_OK) rc = cross_source(y, "y", n, sy);
  if (rc != ICIKT_OK) return rc;
  if (sx->C + sy->C > 2147483647LL) return fail(ICIKT_ERR_BAD_ARG, "too many columns: Cx + Cy > INT32_MAX");
  if (n > tiled_max_n()) return fail(ICIKT_ERR_TOO_LONG, "n exceeds icikt_max_n()");
  if (n_global_na < 0 || (n_global_na > 0 && !global_na)) return fail(ICIKT_ERR_BAD_ARG, "bad global_na");
  if (o.include_diag) return fail(ICIKT_ERR_BAD_ARG, "a cross call has no diagonal: include_diag must be 0");
  if (o.perspective != ICIKT_PERSPECTIVE_GLOBAL && o.perspective != ICIKT_PERSPECTIVE_LOCAL)
    return fail(ICIKT_ERR_BAD_ARG, "a cross call takes the global or the local perspective");
  if (o.kernel != ICIKT_KERNEL_TILED) return fail(ICIKT_ERR_BAD_ARG, "a cross call needs the tiled kernel");
  if (o.want_counts) return fail(ICIKT_ERR_BAD_ARG, "a cross call returns no counts (want_counts)");
  const int64_t ptot = sx->C * sy->C;
  if (ranged ? (o.pair_lo < 0 || o.pair_hi < 0 || o.pair_lo > ptot || o.pair_hi > ptot ||
                (o.pair_hi != 0 && o.pair_lo > o.pair_hi) || (o.pair_hi == 0 && o.pair_lo != 0))
             : (o.pair_lo != 0 || o.pair_hi != 0))
    return fail(ICIKT_ERR_BAD_ARG, ranged ? "pair_lo/pair_hi out of [0, Cx * Cy]"
                                          : "this cross call covers all pairs: pair_lo and pair_hi must be 0");
  return ICIKT_OK;
}

// the walk buffers of icikt_cross_pairs and its two result windows (kept with the plan)
static int ensure_cross_buffers(icikt_plan* p) {
  const int rc = ensure_walk_buffers(p);
  if (rc != ICIKT_OK) return rc;
  const size_t win = (size_t)p->P;  // the plan's pair buffers: W pairs and more
  for (auto& res : p->d_cres)
    if (res.reserve(win * (4 * sizeof(double) + sizeof(int32_t))) != cudaSuccess) {
      cudaGetLastError();
      return fail(ICIKT_ERR_ALLOC, "device allocation of the cross call's result windows failed");
    }
  return ICIKT_OK;
}

// icikt_cross_pairs' walk over pairs [first, last) of `order` (the cross order), into caller arrays indexed from 0 =
// first: per window, the results move off the plan's pair buffers into d_cres[b] on the compute stream (the next
// window's K3 overwrites those buffers), and the host copies them from there into the caller's arrays on the copy
// stream while the next window computes.
template <class Order>
static int cross_pair_walk(icikt_plan* p, const Order& order, int64_t first, int64_t last, int64_t W, double* raw,
                           double* pvalue, double* taumax, double* completeness, int32_t* status, WalkTotals& tot,
                           float& d2h_ms) {
  const size_t win = (size_t)p->P;
  const double* d_field[4] = {p->d_tau, p->d_p, p->d_tm, p->d_comp};
  double* host_field[4] = {raw, pvalue, taumax, completeness};
  auto select = [&](int64_t, int b, const PairUnit*, int64_t, int64_t n_slots) -> int {
    double* to = reinterpret_cast<double*>(p->d_cres[b].get());
    for (int f = 0; f < 4; ++f)
      if (host_field[f])
        CK(cudaMemcpyAsync(to + f * win, d_field[f], sizeof(double) * (size_t)n_slots, cudaMemcpyDeviceToDevice, p->stream));
    if (status)
      CK(cudaMemcpyAsync(to + 4 * win, p->d_status, sizeof(int32_t) * (size_t)n_slots, cudaMemcpyDeviceToDevice, p->stream));
    return ICIKT_OK;
  };
  auto collect = [&](int64_t w, int b) -> int {
    const int64_t off = w * W, cnt = std::min(W, last - first - off);
    const double* from = reinterpret_cast<const double*>(p->d_cres[b].get());
    CK(cudaEventRecord(p->ev[6], p->copy_stream));
    int r = ICIKT_OK;
    for (int f = 0; f < 4 && r == ICIKT_OK; ++f)
      if (host_field[f])
        r = staged_copy_out(p, host_field[f] + off, from + f * win, sizeof(double) * (size_t)cnt, p->copy_stream);
    if (r == ICIKT_OK && status)
      r = staged_copy_out(p, status + off, from + 4 * win, sizeof(int32_t) * (size_t)cnt, p->copy_stream);
    if (r != ICIKT_OK) return r;
    CK(cudaEventRecord(p->ev[7], p->copy_stream));
    CK(cudaEventSynchronize(p->ev[7]));
    d2h_ms += ev_ms(p->ev[6], p->ev[7]);
    return ICIKT_OK;
  };
  return walk_windows(p, order, first, last, W, tot, select, collect);
}

// The list rows of a cross top-k call, [c_lo, c_hi) of [X | Y] (X's columns come first, so any choice of sides is one
// range), and its sides: x_side rows from 0, y_side rows from Cx - c_lo.
static void cross_topk_sides(const icikt_topk_lists* x_side, const icikt_topk_lists* y_side, int64_t Cx, int64_t Cy,
                             int64_t* c_lo, int64_t* c_hi, std::vector<TopkSide>& sides) {
  *c_lo = x_side ? 0 : Cx;
  *c_hi = y_side ? Cx + Cy : Cx;
  if (x_side) sides.push_back(TopkSide{TopkOut{x_side->index, x_side->n_neighbors, x_side->cor, x_side->raw,
                                               x_side->pvalue, x_side->taumax, x_side->completeness},
                                       0, Cx, (int32_t)Cx, {}, nullptr});
  if (y_side) sides.push_back(TopkSide{TopkOut{y_side->index, y_side->n_neighbors, y_side->cor, y_side->raw,
                                               y_side->pvalue, y_side->taumax, y_side->completeness},
                                       Cx - *c_lo, Cy, 0, {}, nullptr});
}

static int pairwise_completeness_impl(const ColumnSource& s, int64_t n, int64_t C, const double* global_na,
                                      int32_t n_global_na, int32_t device, const int32_t* pi, const int32_t* pj,
                                      int64_t P, int32_t* missing, double* completeness, double* matrix) {
  if ((!s.csc() && (!s.data || s.ld < n)) || n < 1 || C < 1) return fail(ICIKT_ERR_BAD_ARG, "bad matrix arguments");
  if ((pi == nullptr) != (pj == nullptr)) return fail(ICIKT_ERR_BAD_ARG, "pi and pj must both be given");
  if (n_global_na < 0 || (n_global_na > 0 && !global_na)) return fail(ICIKT_ERR_BAD_ARG, "bad global_na");
  if (matrix && pi) return fail(ICIKT_ERR_BAD_ARG, "the matrix output covers all pairs; pass pi = pj = NULL");
  if (!pi) P = tri_pairs(C) + C;
  if (pi)
    for (int64_t k = 0; k < P; ++k)
      if (pi[k] < 0 || pi[k] >= C || pj[k] < 0 || pj[k] >= C) return fail(ICIKT_ERR_BAD_ARG, "pair index out of range");
  int rc = select_device(device);
  if (rc != ICIKT_OK) return rc;
  // R/utils.R:6-15: NA and Inf entries of global_na select classes, the rest are literals
  double lit[64];
  int nlit = 0, na_nan = 0, na_inf = 0;
  for (int i = 0; i < n_global_na; ++i) {
    const double v = global_na[i];
    if (std::isnan(v)) { na_nan = 1; continue; }
    if (std::isinf(v)) { na_inf = 1; continue; }
    if (nlit == 64) return fail(ICIKT_ERR_BAD_ARG, "more than 64 global_na literals");
    lit[nlit++] = v;
  }
  const int64_t words = (n + 31) / 32;
  const bool per_pair = missing || completeness;
  struct Buffers {
    Stream stream;  // released after the buffers
    DeviceArray<double> data, lit, comp, mat, values;
    DeviceArray<uint32_t> bits;
    DeviceArray<int32_t> pi, pj, miss, rowidx;
    DeviceArray<int64_t> colptr;
    ~Buffers() {
      if (stream) cudaStreamSynchronize(stream);  // no copy still reads the caller's arrays after an error
    }
  } b;
  CK(b.stream.create());
  CK(b.data.reserve((size_t)n * C));
  CK(b.lit.reserve(64));
  CK(b.bits.reserve((size_t)words * C));
  if (s.csc()) {  // the stored entries, expanded into the dense matrix on the device
    const int64_t nnz = s.colptr[C];
    CK(b.colptr.reserve((size_t)C + 1));
    CK(b.rowidx.reserve((size_t)nnz));
    CK(b.values.reserve((size_t)nnz));
    CK(cudaMemcpyAsync(b.colptr.get(), s.colptr, sizeof(int64_t) * (size_t)(C + 1), cudaMemcpyHostToDevice, b.stream));
    if (nnz) {
      CK(cudaMemcpyAsync(b.rowidx.get(), s.rowidx, sizeof(int32_t) * (size_t)nnz, cudaMemcpyHostToDevice, b.stream));
      CK(cudaMemcpyAsync(b.values.get(), s.values, sizeof(double) * (size_t)nnz, cudaMemcpyHostToDevice, b.stream));
    }
    if (launch_csc_expand(b.colptr.get(), b.rowidx.get(), b.values.get(), n, 0, C, b.data.get(), b.stream) < 0)
      return launch_fail("CSC expansion kernel");
  } else {
    CK(cudaMemcpy2DAsync(b.data.get(), sizeof(double) * n, s.data, sizeof(double) * s.ld, sizeof(double) * n, (size_t)C,
                         cudaMemcpyHostToDevice, b.stream));
  }
  if (nlit) CK(cudaMemcpyAsync(b.lit.get(), lit, sizeof(double) * nlit, cudaMemcpyHostToDevice, b.stream));
  if (launch_missing_bits(b.data.get(), n, n, C, b.lit.get(), nlit, na_nan, na_inf, b.bits.get(), words, b.stream) < 0)
    return launch_fail("missing-mask kernel");
  if (per_pair) {
    if (pi) {
      CK(b.pi.reserve((size_t)P));
      CK(b.pj.reserve((size_t)P));
      CK(cudaMemcpyAsync(b.pi.get(), pi, sizeof(int32_t) * P, cudaMemcpyHostToDevice, b.stream));
      CK(cudaMemcpyAsync(b.pj.get(), pj, sizeof(int32_t) * P, cudaMemcpyHostToDevice, b.stream));
    }
    if (missing) CK(b.miss.reserve((size_t)P));
    if (completeness) CK(b.comp.reserve((size_t)P));
    if (launch_pair_missing(b.bits.get(), words, n, C, b.pi.get(), b.pj.get(), P, b.miss.get(), b.comp.get(), b.stream) < 0)
      return launch_fail("pair completeness kernel");
    if (missing) CK(cudaMemcpyAsync(missing, b.miss.get(), sizeof(int32_t) * P, cudaMemcpyDeviceToHost, b.stream));
    if (completeness) CK(cudaMemcpyAsync(completeness, b.comp.get(), sizeof(double) * P, cudaMemcpyDeviceToHost, b.stream));
  }
  if (matrix) {
    CK(b.mat.reserve((size_t)C * C));
    if (launch_missing_matrix(b.bits.get(), words, n, C, b.mat.get(), b.stream) < 0)
      return launch_fail("completeness matrix kernel");
    CK(cudaMemcpyAsync(matrix, b.mat.get(), sizeof(double) * C * C, cudaMemcpyDeviceToHost, b.stream));
  }
  CK(cudaStreamSynchronize(b.stream));
  return ICIKT_OK;
}

extern "C" {

int icikt_pairwise_completeness(const double* data, int64_t n, int64_t C, int64_t ld, const double* global_na,
                                int32_t n_global_na, int32_t device, const int32_t* pi, const int32_t* pj,
                                int64_t P, int32_t* missing, double* completeness, double* matrix) {
  return pairwise_completeness_impl(dense_source(data, ld, C), n, C, global_na, n_global_na, device, pi, pj, P, missing,
                                    completeness, matrix);
}

int icikt_pairwise_completeness_csc(const int64_t* colptr, const int32_t* rowidx, const double* values, int64_t n,
                                    int64_t C, const double* global_na, int32_t n_global_na, int32_t device,
                                    const int32_t* pi, const int32_t* pj, int64_t P, int32_t* missing,
                                    double* completeness, double* matrix) {
  const int rc = check_csc(colptr, rowidx, values, n, C);
  if (rc != ICIKT_OK) return rc;
  return pairwise_completeness_impl(csc_source(colptr, rowidx, values, C), n, C, global_na, n_global_na, device, pi, pj,
                                    P, missing, completeness, matrix);
}

}  // extern "C"

namespace {

// One multi-device job: worker k (one host thread per device) owns the k-th contiguous slice of the
// pair order.  Sharded preprocessing: if every pair of devices can reach each other directly (NVLink /
// NVSwitch), device k uploads only its slice of the columns over its own PCIe link, runs K1 on that
// slice and pulls the other slices of the per-column TABLES from its peers (an all-gather by peer
// copies: K1 is not replicated and the raw matrix never travels between devices); otherwise every
// device uploads the whole matrix and preprocesses all columns.  A cross call's job holds [X | Y]: src is X, y is Y
// (placed from column src.C on), C = Cx + Cy, and the slices cover pairs [first, first + ptot) of the cross order.  A
// pair-list job (one worker) computes the ptot pairs (pi[k], pj[k]).
struct MultiJob {
  ColumnSource src;
  const ColumnSource* y = nullptr;
  const int32_t *pi = nullptr, *pj = nullptr;
  int64_t n, C;
  const double* global_na;
  int32_t n_global_na;
  icikt_opts base;
  const int32_t* devices;
  int n_devices;
  int64_t first = 0, ptot;
  bool peers_ok = false;  // every pair of distinct ordinals has peer access
  bool gather = false;    // sharded K1 + peer gather of the tables
  HostBarrier barrier;
  std::vector<icikt_plan*> peer_plan;
  explicit MultiJob(int nd) : n_devices(nd), barrier(nd), peer_plan((size_t)nd, nullptr) {}
  int device_of(int k) const { return devices ? devices[k] : k; }
  int64_t pair_lo(int k) const { return first + ptot * k / n_devices; }  // slices differ by at most one pair
  int64_t col_lo(int k) const { return C * k / n_devices; }
  bool idle(int k) const { return n_devices > 1 && pair_lo(k + 1) <= pair_lo(k); }  // one of several, without pairs
};

// An all-pairs job over the whole combn order of s (the diagonal included if o.include_diag), its arguments checked.
void all_pairs_job(MultiJob& J, const ColumnSource& s, int64_t n, const double* global_na, int32_t n_global_na,
                   const icikt_opts& o, const int32_t* devices) {
  J.src = s; J.n = n; J.C = s.C; J.global_na = global_na; J.n_global_na = n_global_na;
  J.devices = devices; J.base = o; J.ptot = tri_pairs(s.C) + (o.include_diag ? s.C : 0);
}

// A cross job over pairs [first, last) of the cross order, its arguments checked.  The window plans hold W pairs of
// a slice: the call's pair range is the job's, not theirs.
void cross_job(MultiJob& J, const ColumnSource& sx, const ColumnSource& sy, int64_t n, const double* global_na,
               int32_t n_global_na, const icikt_opts& o, const int32_t* devices, int64_t first, int64_t last) {
  J.src = sx; J.y = &sy; J.n = n; J.C = sx.C + sy.C; J.global_na = global_na; J.n_global_na = n_global_na;
  J.devices = devices; J.base = o; J.base.pair_lo = J.base.pair_hi = 0;
  J.first = first; J.ptot = last - first;
}

void multi_probe_peers(MultiJob& J) {
  bool distinct = true;
  J.peers_ok = true;
  for (int a = 0; a < J.n_devices; ++a)
    for (int b = 0; b < J.n_devices; ++b) {
      if (a == b) continue;
      const int da = J.device_of(a), db = J.device_of(b);
      if (da == db) { distinct = false; continue; }
      int ok = 0;
      if (cudaDeviceCanAccessPeer(&ok, da, db) != cudaSuccess || !ok) J.peers_ok = false;
    }
  cudaGetLastError();
  // ICIKT_FORCE_PEER_GATHER: repeated ordinals take gather mode too (a same-device peer copy is a device-to-device
  // copy), so that one GPU runs the sharded column phase
  J.gather = J.n_devices >= 2 && (distinct || std::getenv("ICIKT_FORCE_PEER_GATHER")) && J.peers_ok &&
             J.C >= J.n_devices && J.ptot >= J.n_devices && !std::getenv("ICIKT_NO_PEER_GATHER");
}

int enable_peers(const MultiJob& J, int k) {
  for (int j = 0; j < J.n_devices; ++j) {
    if (J.device_of(j) == J.device_of(k)) continue;
    const cudaError_t e = cudaDeviceEnablePeerAccess(J.device_of(j), 0);
    if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) return cuda_fail(e, "cudaDeviceEnablePeerAccess");
    cudaGetLastError();
  }
  return ICIKT_OK;
}

// The peer phase of worker k, once its part is on its device (rc: how that went): it publishes its plan p, or null
// if it failed, and waits until every worker has.  If every worker succeeded it enables peer access and runs body(),
// which reads the other workers' buffers in place (J.peer_plan); otherwise it fails with `peer_failed`.  Then it waits
// until every worker is done, so that nobody's buffers are touched (or freed) while a peer still reads them.  Every
// worker passes both barriers whatever happened to it, so nobody is left waiting.
template <class Body>
int peer_phase(MultiJob& J, int k, icikt_plan* p, int rc, const char* peer_failed, Body&& body) {
  J.peer_plan[(size_t)k] = (rc == ICIKT_OK) ? p : nullptr;
  J.barrier.wait();
  bool all_ok = true;
  for (int j = 0; j < J.n_devices; ++j) all_ok = all_ok && J.peer_plan[(size_t)j] != nullptr;
  if (rc == ICIKT_OK && !all_ok) rc = fail(ICIKT_ERR_CUDA, peer_failed);
  if (rc == ICIKT_OK) rc = enable_peers(J, k);
  if (rc == ICIKT_OK) rc = body();
  J.barrier.wait();
  return rc;
}

// The column phase of worker k on its plan p (rc: how getting the plan went): sharded K1 and the peer gather of the
// tables in gather mode, otherwise the upload and K1 of all columns (skipped by an idle worker).  A cross job's
// columns are those of [X | Y]: a shard that straddles column Cx uploads X's part, then Y's (upload_span).
int multi_worker_columns(MultiJob& J, int k, icikt_plan* p, int rc) {
  if (!J.gather) return J.idle(k) || rc != ICIKT_OK ? rc : window_columns(p, J.src, J.global_na, J.n_global_na, J.y);
  int x_launches = 0;
  if (rc == ICIKT_OK) rc = upload_span(p, J.src, J.y, J.col_lo(k), J.col_lo(k + 1), &x_launches);
  if (rc == ICIKT_OK) rc = icikt_plan_columns_range(p, J.global_na, J.n_global_na, J.col_lo(k), J.col_lo(k + 1));
  if (rc == ICIKT_OK) p->tm.n_launches += x_launches;
  if (rc == ICIKT_OK && cudaStreamSynchronize(p->stream) != cudaSuccess) rc = cuda_fail(cudaGetLastError(), "column slice");
  return peer_phase(J, k, p, rc, "a peer device failed to preprocess its slice", [&]() -> int {
    const int dev = J.device_of(k);
    icikt_table mine[ICIKT_MAX_TABLES], theirs[ICIKT_MAX_TABLES];
    const int nt = icikt_plan_tables(p, mine, ICIKT_MAX_TABLES);
    int r = ICIKT_OK;
    for (int j = 0; j < J.n_devices && r == ICIKT_OK; ++j) {
      if (j == k) continue;
      icikt_plan_tables(J.peer_plan[(size_t)j], theirs, ICIKT_MAX_TABLES);
      for (int t = 0; t < nt && r == ICIKT_OK; ++t) {
        const size_t off = (size_t)J.col_lo(j) * (size_t)mine[t].bytes_per_column;
        const size_t len = (size_t)(J.col_lo(j + 1) - J.col_lo(j)) * (size_t)mine[t].bytes_per_column;
        if (len && cudaMemcpyPeerAsync(static_cast<unsigned char*>(mine[t].ptr) + off, dev,
                                       static_cast<const unsigned char*>(theirs[t].ptr) + off, J.device_of(j), len,
                                       p->stream) != cudaSuccess)
          r = cuda_fail(cudaGetLastError(), "cudaMemcpyPeerAsync");
      }
    }
    if (r == ICIKT_OK) r = icikt_plan_columns_finish(p);
    if (r == ICIKT_OK && cudaStreamSynchronize(p->stream) != cudaSuccess) r = cuda_fail(cudaGetLastError(), "peer gather");
    return r;
  });
}

// The cached plans of a per-pair job's workers, as window_slots: one worker takes g_cached, several one slot each.
icikt_plan** pair_slots(const MultiJob& J) { return J.n_devices == 1 ? &g_cached : g_cached_multi; }

// The per-pair and matrix calls as a job over the caller's pair range (0, 0: all pairs) or pair list, with the checks
// of their arguments that need no device.
int pairs_job(MultiJob& J, const ColumnSource& s, int64_t n, int64_t C, const double* global_na, int32_t n_global_na,
              const int32_t* pi, const int32_t* pj, int64_t P, const icikt_opts& o, const int32_t* devices) {
  if (n < 1 || C < 1) return fail(ICIKT_ERR_BAD_ARG, "n and C must be >= 1");
  if (C > 2147483647LL) return fail(ICIKT_ERR_BAD_ARG, "too many columns");
  if (!s.csc() && s.ld < n) return fail(ICIKT_ERR_BAD_ARG, "bad upload arguments");
  const int64_t all = tri_pairs(C) + (o.include_diag ? C : 0);
  const int64_t lo = o.pair_lo, hi = (o.pair_lo == 0 && o.pair_hi == 0) ? all : o.pair_hi;
  if (!pi && (lo < 0 || hi > all || lo > hi)) return fail(ICIKT_ERR_BAD_ARG, "pair_lo/pair_hi out of range");
  all_pairs_job(J, s, n, global_na, n_global_na, o, devices);
  J.pi = pi; J.pj = pj;
  J.first = pi ? 0 : lo;
  J.ptot = pi ? P : hi - lo;
  return ICIKT_OK;
}

// A lone worker over the whole pair order of a large input runs the pipelined call (run_staged).
bool job_staged(const MultiJob& J) {
  return J.n_devices == 1 && !J.pi && J.first == 0 && J.ptot == tri_pairs(J.C) + (J.base.include_diag ? J.C : 0) &&
         want_staged(J.n, J.C, J.base);
}

// the per-pair output arrays of a call, indexed from 0 = the job's first pair
struct PairArrays {
  double *raw, *pvalue, *taumax, *completeness;
  int32_t* status;
  int64_t* counts;
};

// Worker k of a per-pair job: its plan (slots[k]; a pair list's is built from J.pi / J.pj), the column phase and the
// pair kernel + epilogue, then, given `to`, the download of its slice at its offset from J.first (mx: the slice's
// maximum taumax); without `to` the results stay on its device.  `staged` (job_staged): all of it as the pipelined
// call.  An idle worker only takes part in the column phase.
int pairs_worker(MultiJob& J, int k, icikt_plan** slots, bool staged, const PairArrays* to, icikt_plan** out,
                 double* mx) {
  icikt_opts o = J.base;
  o.device = J.device_of(k);
  o.pair_lo = staged ? 0 : J.pair_lo(k);  // a staged plan covers the whole order as 0, 0
  o.pair_hi = staged ? 0 : J.pair_lo(k + 1);
  int rc;
  if (J.pi) {
    rc = plan_create_impl(out, J.n, J.C, J.pi, J.pj, J.ptot, &o, false);
    slots[k] = *out;
  } else {
    rc = cached_plan(slots[k], J.n, J.C, o, staged, out);
  }
  icikt_plan* p = *out;
  if (staged) {
    const PairArrays d = to ? *to : PairArrays{};
    return rc != ICIKT_OK ? rc : run_staged(p, J.src, J.global_na, J.n_global_na, to != nullptr, d.raw, d.pvalue,
                                            d.taumax, d.completeness, d.status, d.counts, mx);
  }
  rc = multi_worker_columns(J, k, p, rc);
  if (rc == ICIKT_OK && !J.idle(k)) rc = icikt_plan_pairs(p);
  if (rc != ICIKT_OK || J.idle(k) || !to) return rc;
  const int64_t off = J.pair_lo(k) - J.first;
  auto at = [off](auto* a, int64_t per_pair = 1) { return a ? a + off * per_pair : a; };
  return icikt_plan_download(p, at(to->raw), at(to->pvalue), at(to->taumax), at(to->completeness), at(to->status),
                             at(to->counts, ICIKT_NCOUNTS), mx);
}

struct MultiWork {
  int rc = ICIKT_OK;
  std::string err;
  double mx = std::nan("");
  icikt_timings tm{};
  unsigned long long hist[16] = {};
};

int multi_collect(const std::vector<MultiWork>& work, double* max_taumax, icikt_timings* timings) {
  double mx = std::nan("");
  icikt_timings slowest{};
  for (const MultiWork& w : work) {
    if (w.rc != ICIKT_OK) return fail(w.rc, w.err);
    if (w.mx == w.mx && !(mx >= w.mx)) mx = w.mx;
    if (w.tm.total_ms >= slowest.total_ms) {
      const int launches = slowest.n_launches + w.tm.n_launches;
      slowest = w.tm;
      slowest.n_launches = launches;
    } else {
      slowest.n_launches += w.tm.n_launches;
    }
  }
  if (max_taumax) *max_taumax = mx;
  if (timings) *timings = slowest;
  return ICIKT_OK;
}

// The workers of J: w.rc = body(k, w) for worker k, on the calling thread when there is one worker, on a thread each
// otherwise.  A worker that fails keeps its message and drops its cached plan slots[k]; then multi_collect.  The
// caller holds g_cache_mu (the cached plans are not re-entrant).
template <class Body>
int run_workers(const MultiJob& J, icikt_plan** slots, std::vector<MultiWork>& work, double* max_taumax,
                icikt_timings* timings, Body&& body) {
  work.assign((size_t)J.n_devices, MultiWork{});
  auto run = [&](int k) {
    MultiWork& w = work[(size_t)k];
    w.rc = body(k, w);
    if (w.rc != ICIKT_OK) {
      w.err = g_err;  // thread-local message of this worker
      icikt_plan_destroy(slots[k]);  // waits for whatever the failed worker left in flight
      slots[k] = nullptr;
    }
  };
  if (J.n_devices == 1) {
    run(0);
  } else {
    std::vector<std::thread> threads;
    for (int k = 0; k < J.n_devices; ++k) threads.emplace_back(run, k);
    for (auto& t : threads) t.join();
  }
  return multi_collect(work, max_taumax, timings);
}

// The per-pair calls: icikt_all_pairs and icikt_pair_list are the job of one worker on opts->device, the _multi twins
// that of the caller's devices.
int pairs_impl(const ColumnSource& s, int64_t n, int64_t C, const double* global_na, int32_t n_global_na,
               const int32_t* pi, const int32_t* pj, int64_t P, icikt_opts o, const int32_t* devices, int32_t n_devices,
               const PairArrays& to, double* max_taumax, icikt_timings* timings) {
  if ((!s.data && !s.csc()) || !to.raw) return fail(ICIKT_ERR_BAD_ARG, "data and raw must not be NULL");
  if (n_devices < 1 || n_devices > 64) return fail(ICIKT_ERR_BAD_ARG, "n_devices must be 1..64");
  o.want_counts = to.counts ? 1 : 0;
  MultiJob J(n_devices);
  int rc = pairs_job(J, s, n, C, global_na, n_global_na, pi, pj, P, o, devices);
  if (rc != ICIKT_OK) return rc;
  std::lock_guard<std::mutex> lock(g_cache_mu);  // the cached plans are not re-entrant
  multi_probe_peers(J);
  const bool staged = job_staged(J);
  icikt_plan* list_plan = nullptr;  // a pair list's plan is freed at the end of the call
  icikt_plan** slots = pi ? &list_plan : pair_slots(J);
  std::vector<MultiWork> work;
  rc = run_workers(J, slots, work, max_taumax, timings, [&](int k, MultiWork& w) -> int {
    icikt_plan* p = nullptr;
    int r = pairs_worker(J, k, slots, staged, &to, &p, &w.mx);
    if (r == ICIKT_OK && timings && !J.idle(k)) r = icikt_plan_timings(p, &w.tm);
    return r;
  });
  icikt_plan_destroy(list_plan);
  return rc;
}

// The matrix calls: one worker computes its pairs and fills the matrices (icikt_plan_download_matrices); several, with
// peer access between them, fill a block of columns each from every device's results (matrix_block_fill_kernel).
int matrices_impl(const ColumnSource& s, int64_t n, int64_t C, const double* global_na, int32_t n_global_na,
                  const int32_t* pi, const int32_t* pj, int64_t P, icikt_opts o, const int32_t* devices,
                  int32_t n_devices, int32_t scale_max, int32_t diag_good, const int32_t* n_good, double* cor,
                  double* raw, double* pvalue, double* taumax, double* completeness, int64_t* status_counts,
                  double* max_taumax, icikt_timings* timings) {
  if (!pi) o.include_diag = diag_good ? 0 : 1;  // setup_comparisons, R/kendalltau.R:191-194
  o.want_counts = 0;
  MultiJob J(n_devices);
  int rc = pairs_job(J, s, n, C, global_na, n_global_na, pi, pj, P, o, devices);
  if (rc != ICIKT_OK) return rc;
  std::lock_guard<std::mutex> lock(g_cache_mu);  // the cached plans are not re-entrant
  multi_probe_peers(J);
  // devices that cannot read each other's results, or fewer pairs or columns than devices: one worker on devices[0]
  if (!J.peers_ok || J.ptot < J.n_devices || C < J.n_devices) J.n_devices = 1;
  const bool staged = job_staged(J);
  icikt_plan* list_plan = nullptr;  // a pair list's plan is freed at the end of the call
  icikt_plan** slots = pi ? &list_plan : pair_slots(J);
  const int n_dev = J.n_devices;
  double* outs[5] = {cor, raw, pvalue, taumax, completeness};
  std::vector<MultiWork> work;
  std::vector<int32_t> good((size_t)C, 0);
  if (n_good) std::copy(n_good, n_good + C, good.begin());
  rc = run_workers(J, slots, work, max_taumax, timings, [&](int k, MultiWork& w) -> int {
    icikt_plan* p = nullptr;
    w.rc = pairs_worker(J, k, slots, staged, nullptr, &p, nullptr);
    if (n_dev == 1) {  // the whole matrices from this worker's results
      if (w.rc == ICIKT_OK)
        w.rc = icikt_plan_download_matrices(p, scale_max, diag_good, n_good, cor, raw, pvalue, taumax, completeness,
                                            status_counts, &w.mx);
      if (w.rc == ICIKT_OK && timings) w.rc = icikt_plan_timings(p, &w.tm);
      return w.rc;
    }
    unsigned long long bits = 0;
    if (w.rc == ICIKT_OK) {
      if (cudaMemcpyAsync(&bits, p->d_maxbits, sizeof(bits), cudaMemcpyDeviceToHost, p->stream) != cudaSuccess ||
          cudaStreamSynchronize(p->stream) != cudaSuccess)
        w.rc = cuda_fail(cudaGetLastError(), "pair kernel");
    }
    if (w.rc == ICIKT_OK && bits) std::memcpy(&w.mx, &bits, sizeof(bits));
    if (w.rc == ICIKT_OK && k == 0 && diag_good && !n_good) {  // n_good = n - missing rows (R/kendalltau.R:165)
      w.rc = icikt_plan_column_info(p, good.data());
      for (int64_t c = 0; c < C && w.rc == ICIKT_OK; ++c) good[(size_t)c] = (int32_t)n - good[(size_t)c];
    }
    return peer_phase(J, k, p, w.rc, "a peer device failed to compute its pairs", [&]() -> int {
      double mx = std::nan("");
      for (const MultiWork& v : work)
        if (v.mx == v.mx && !(mx >= v.mx)) mx = v.mx;
      const int64_t c_lo = J.col_lo(k), c_hi = J.col_lo(k + 1);
      const size_t blk = (size_t)C * (size_t)(c_hi - c_lo);
      CK(cudaSetDevice(p->device));
      int r = ensure_matrix_buffers(p, 5 * blk, "the result matrix block");
      if (r == ICIKT_OK) r = ensure_stage(p);
      if (r != ICIKT_OK) return r;
      CK(cudaEventRecord(p->ev[6], p->stream));
      CK(cudaMemsetAsync(p->d_hist.get(), 0, 16 * sizeof(unsigned long long), p->stream));
      BlockFill f{};
      f.n_dev = n_dev;
      for (int j = 0; j < n_dev; ++j) {
        const icikt_plan* q = J.peer_plan[(size_t)j];
        f.tau[j] = q->d_tau; f.pvalue[j] = q->d_p; f.taumax[j] = q->d_tm; f.completeness[j] = q->d_comp;
        f.status[j] = q->d_status;
        f.pair_lo[j] = J.pair_lo(j);
      }
      f.pair_lo[n_dev] = J.ptot;
      f.n = n; f.C = C; f.c_lo = c_lo; f.c_hi = c_hi;
      f.scale_max = scale_max != 0; f.diag_good = diag_good != 0;
      f.max_taumax = mx;
      f.n_good = p->d_ngood.get();
      int best = 1;
      if (diag_good) {
        CK(cudaMemcpyAsync(p->d_ngood.get(), good.data(), sizeof(int32_t) * (size_t)C, cudaMemcpyHostToDevice, p->stream));
        best = 0;
        for (int64_t c = 0; c < C; ++c) best = std::max(best, good[(size_t)c]);
      }
      f.best_good = best;
      for (int q = 0; q < 5; ++q) f.m[q] = outs[q] ? p->d_mat.get() + (size_t)q * blk : nullptr;
      f.hist = p->d_hist.get();
      if (launch_matrix_block_fill(f, p->stream) < 0) return launch_fail("matrix block fill kernel");
      for (int q = 0; q < 5; ++q)
        if (outs[q] && blk) {
          const int r2 = staged_copy_out(p, outs[q] + (size_t)c_lo * (size_t)C, f.m[q], sizeof(double) * blk, p->stream);
          if (r2 != ICIKT_OK) return r2;
        }
      CK(cudaMemcpyAsync(w.hist, p->d_hist.get(), sizeof(w.hist), cudaMemcpyDeviceToHost, p->stream));
      CK(cudaEventRecord(p->ev[7], p->stream));
      CK(cudaStreamSynchronize(p->stream));
      return icikt_plan_timings(p, &w.tm);
    });
  });
  icikt_plan_destroy(list_plan);
  if (rc != ICIKT_OK || n_dev == 1) return rc;
  if (status_counts) {
    int64_t bad = 0;
    for (int q = 1; q < ICIKT_NSTATUS; ++q) {
      status_counts[q] = 0;
      for (const MultiWork& w : work) status_counts[q] += (int64_t)w.hist[q];
      bad += status_counts[q];
    }
    status_counts[0] = J.ptot - bad;
  }
  return ICIKT_OK;
}

// ---- the windowed calls (filtered, top-k and cross) on one device or several: the pair order sliced as in
// icikt_all_pairs_multi, every slice walked window by window on its device, the per-device results combined exactly.
// A single-device call is the job of one worker, run on the calling thread.

icikt_opts opts_or_default(const icikt_opts* opts) {
  icikt_opts o;
  if (opts) o = *opts; else icikt_default_opts(&o);
  return o;
}

int check_window_devices(int32_t n_devices) {
  if (n_devices < 1 || n_devices > kMaxMatrixDevices) return fail(ICIKT_ERR_BAD_ARG, "n_devices must be 1..16");
  return ICIKT_OK;
}

// The matrix x of an all-pairs call that takes an icikt_input, and the arguments the windowed calls share, checked
// before any device is touched.
int check_all_pairs_input(const icikt_input* x, int64_t n, const double* global_na, int32_t n_global_na,
                          const icikt_opts& o, int32_t n_devices, ColumnSource* s) {
  int rc = n < 1 ? fail(ICIKT_ERR_BAD_ARG, "n and C must be >= 1") : cross_source(x, "x", n, s);
  if (rc == ICIKT_OK) rc = check_window_args(*s, n, s->C, global_na, n_global_na, o);
  return rc == ICIKT_OK ? check_window_devices(n_devices) : rc;
}

// The cached window plans of J's workers: one worker takes the single-device slot, several take one slot each, so
// that one-device and multi-device calls alternated on the same data do not reallocate each other's plans.
icikt_plan** window_slots(const MultiJob& J) { return J.n_devices == 1 ? &g_cached_edges : g_cached_wmulti; }

// Worker k of a windowed job up to its window walk: its window plan (windows of min(ICIKT_EDGE_WINDOW, its slice)
// pairs and at least one) and the column phase.
int window_multi_worker(MultiJob& J, int k, icikt_plan** out) {
  icikt_opts o = J.base;
  o.device = J.device_of(k);
  o.pair_hi = std::max<int64_t>(1, std::min(edge_window(), J.pair_lo(k + 1) - J.pair_lo(k)));  // pair_lo is 0
  int rc = cached_plan(window_slots(J)[k], J.n, J.C, o, false, out);
  rc = multi_worker_columns(J, k, *out, rc);
  if (rc == ICIKT_OK) CK(cudaSetDevice((*out)->device));
  return rc;
}

// The windowed job J, its arguments checked.  Worker k takes its window plan p and runs the column phase
// (window_multi_worker); walk(k, p, order, lo, hi, tot, d2h_ms) then reserves its buffers and walks its slice [lo, hi)
// of J's pair order (`order`: the cross order of a cross job, the combn order otherwise), d2h_ms receiving the time
// of its copies out, and finish_walk gives its timings.  An idle worker walks nothing.  *M receives the maximum
// taumax over all pairs; a job without pairs walks nothing and leaves *M NaN and the timings zero.
// `merge` (the top-k lists, merged on the devices): devices that cannot read each other's lists make the job one
// worker on devices[0]; of several workers, every one then runs merge(k, p, rc, tm) whatever its rc, and an idle
// worker walks its empty slice too, so that the merge reads empty lists.
template <class Walk>
int run_windows(MultiJob& J, double* M, icikt_timings* timings, Walk&& walk,
                const std::function<int(int, icikt_plan*, int, icikt_timings&)>& merge = nullptr) {
  int rc = select_device(J.device_of(0));
  if (rc != ICIKT_OK) return rc;
  *M = std::nan("");
  if (J.ptot == 0) {  // one column without the diagonal, or an empty cross range: nothing to compute
    if (timings) std::memset(timings, 0, sizeof(*timings));
    return ICIKT_OK;
  }
  std::vector<MultiWork> work;
  std::vector<unsigned long long> bits((size_t)J.n_devices, 0);
  std::lock_guard<std::mutex> lock(g_cache_mu);  // the cached plans are not re-entrant
  multi_probe_peers(J);
  if (merge && !J.peers_ok) J.n_devices = 1;
  rc = run_workers(J, window_slots(J), work, nullptr, timings, [&](int k, MultiWork& w) -> int {
    icikt_plan* p = nullptr;
    int r = window_multi_worker(J, k, &p);
    if (r == ICIKT_OK && (merge || !J.idle(k))) {
      WalkTotals tot;
      float d2h_ms = 0.f;
      const int64_t lo = J.pair_lo(k), hi = J.pair_lo(k + 1);
      auto walk_on = [&](const auto& order) { return walk(k, p, order, lo, hi, tot, d2h_ms); };
      r = J.y ? walk_on(cross_order(J.src.C, J.y->C)) : walk_on(combn_order(p));
      if (r == ICIKT_OK) r = finish_walk(p, tot, d2h_ms, &w.tm);
      bits[(size_t)k] = tot.bits;
    }
    return merge && J.n_devices > 1 ? merge(k, p, r, w.tm) : r;
  });
  if (rc == ICIKT_OK) *M = max_of_bits(*std::max_element(bits.begin(), bits.end()));
  return rc;
}

// The adjusted p-values of the rows held (the _padj calls), once every worker has walked its slice: m is the sum of
// the workers' non-NaN counts; their candidates are gathered on devices[0] (the same device: a device copy; peer
// access between all devices: peer copies; otherwise through pinned host memory), sorted and scanned there once, and
// every row looks its value up there.  m <= 1 leaves the p-values as they are (p.adjust).  Then the rows with
// padj > max_padj go.  dev_ms receives the device time of the gather, sort, scan and lookup.
int padj_gather(const MultiJob& J, std::vector<PadjPart>& parts, int dev, int64_t K, unsigned long long** all,
                DeviceArray<unsigned long long>& own) {
  PadjPart& first = parts[0];
  int64_t at = 0;
  size_t k0 = 0;
  if (first.device == dev && (int64_t)first.d_keys.size() >= K) {  // the first worker's buffer takes the others' candidates
    *all = first.d_keys.get();
    at = first.K;
    k0 = 1;
  } else {
    if (own.reserve((size_t)K) != cudaSuccess) {
      cudaGetLastError();
      return fail(ICIKT_ERR_ALLOC, "device allocation for the " + std::to_string(K) + " p-value candidates failed");
    }
    *all = own.get();
  }
  PinnedArray<unsigned long long> stage;
  const size_t chunk = 4u << 20;  // keys per staged piece (32 MB)
  int rc = ICIKT_OK;
  for (size_t k = k0; k < parts.size() && rc == ICIKT_OK; ++k) {
    PadjPart& pt = parts[k];
    const size_t bytes = sizeof(unsigned long long) * (size_t)pt.K;
    cudaError_t e = cudaSuccess;
    if (!pt.K) continue;
    if (pt.device == dev) {
      e = cudaMemcpy(*all + at, pt.d_keys.get(), bytes, cudaMemcpyDeviceToDevice);
    } else if (J.peers_ok) {
      e = cudaMemcpyPeer(*all + at, dev, pt.d_keys.get(), pt.device, bytes);
    } else {
      if ((e = stage.reserve(chunk)) != cudaSuccess) break;
      for (int64_t o = 0; o < pt.K && e == cudaSuccess; o += (int64_t)chunk) {
        const size_t b = sizeof(unsigned long long) * std::min<size_t>(chunk, (size_t)(pt.K - o));
        if ((e = cudaSetDevice(pt.device)) == cudaSuccess) e = cudaMemcpy(stage.get(), pt.d_keys.get() + o, b, cudaMemcpyDeviceToHost);
        if (e == cudaSuccess && (e = cudaSetDevice(dev)) == cudaSuccess)
          e = cudaMemcpy(*all + at + o, stage.get(), b, cudaMemcpyHostToDevice);
      }
    }
    if (e != cudaSuccess) rc = cuda_fail(e, "gathering the p-value candidates");
    at += pt.K;
    cudaSetDevice(pt.device);  // the part is gathered: free its buffers on their device now
    pt.d_keys.reset();
    pt.d_cnt.reset();
    pt.h_cnt.reset();
    pt.device = -1;
    cudaSetDevice(dev);
  }
  return rc;
}

int padj_finish(const MultiJob& J, std::vector<PadjPart>& parts, const icikt_padj_filter& a, icikt_edges* res,
                float* dev_ms) {
  int64_t m = 0, K = 0;
  for (const PadjPart& pt : parts) {
    m += pt.m;
    K += pt.K;
  }
  res->n_tests = m;
  std::vector<EdgeRow>& rows = res->rows;
  std::vector<double>& padj = res->padj;
  const int64_t R = (int64_t)rows.size();
  try {
    padj.resize((size_t)R);
  } catch (const std::bad_alloc&) {
    return fail(ICIKT_ERR_ALLOC, "out of host memory for the adjusted p-values");
  }
  *dev_ms = 0.f;
  if (m <= 1) {
    for (int64_t r = 0; r < R; ++r) padj[(size_t)r] = rows[(size_t)r].pvalue;
  } else if (R > 0) {
    const int dev = J.device_of(0);
    CK(cudaSetDevice(dev));
    Event ev[2];
    CK(ev[0].create());
    CK(ev[1].create());
    CK(cudaEventRecord(ev[0], 0));
    unsigned long long* all = nullptr;
    DeviceArray<unsigned long long> own;
    int rc = padj_gather(J, parts, dev, K, &all, own);
    if (rc != ICIKT_OK) return rc;
    const double q = a.method == ICIKT_PADJ_BY ? padj_by_q(m) : 0.0;
    unsigned long long* sorted = nullptr;
    double* vals = nullptr;
    DeviceArray<unsigned long long> alt;
    DeviceArray<double> d_p;
    if (alt.reserve((size_t)K) != cudaSuccess || d_p.reserve(2 * (size_t)R) != cudaSuccess) {
      cudaGetLastError();
      return fail(ICIKT_ERR_ALLOC, "device allocation for sorting " + std::to_string(K) + " p-value candidates failed");
    }
    std::vector<double> p;
    try {
      p.resize((size_t)R);
    } catch (const std::bad_alloc&) {
      return fail(ICIKT_ERR_ALLOC, "out of host memory for the adjusted p-values");
    }
    for (int64_t r = 0; r < R; ++r) p[(size_t)r] = rows[(size_t)r].pvalue;
    CK(padj_sort_scan(all, alt.get(), K, m, a.method, q, &sorted, &vals, 0));
    CK(cudaMemcpy(d_p.get(), p.data(), sizeof(double) * (size_t)R, cudaMemcpyHostToDevice));
    CK(padj_lookup(sorted, vals, K, a.method, d_p.get(), R, d_p.get() + R, 0));
    CK(cudaMemcpy(padj.data(), d_p.get() + R, sizeof(double) * (size_t)R, cudaMemcpyDeviceToHost));
    CK(cudaEventRecord(ev[1], 0));
    CK(cudaEventSynchronize(ev[1]));
    *dev_ms = ev_ms(ev[0], ev[1]);
  }
  const double t = a.max_padj;
  if (t == t) {
    size_t w = 0;
    for (size_t r = 0; r < rows.size(); ++r)
      if (padj[r] <= t) {
        rows[w] = rows[r];
        padj[w++] = padj[r];
      }
    rows.resize(w);
    padj.resize(w);
  }
  return ICIKT_OK;
}

// The filtered call over the devices of J, its arguments checked: every worker walks its slice against the shared
// EdgeHeld, then the rows are joined in worker order (the slices are contiguous and in order, so are the rows; the
// first worker's rows are moved, not copied) and edge_result trims them with the final maximum.  With `adjust`
// (the _padj calls), every worker also keeps its candidates, and padj_finish gives the rows their adjusted values.
int edges_run(MultiJob& J, const icikt_edge_filter& f0, icikt_edges** out, double* max_taumax, icikt_timings* timings,
              const icikt_padj_filter* adjust = nullptr) {
  // The candidate bound: every row with padj <= max_padj has p <= max_padj (icikt_padj.cuh).  A max_padj >= 1 keeps
  // every row, as does NaN.  The rows take it as one more p-value bound.
  icikt_edge_filter f = f0;
  std::vector<PadjPart> parts(adjust ? (size_t)J.n_devices : 0);
  if (adjust) {
    const double b = adjust->max_padj < 1.0 ? adjust->max_padj : std::nan("");
    for (PadjPart& pt : parts) pt.bound = b;
    if (b == b && !(f.max_pvalue <= b)) f.max_pvalue = b;
  }
  std::vector<std::vector<EdgeRow>> rows((size_t)J.n_devices);
  EdgeHeld held;
  double M;
  int rc = run_windows(J, &M, timings, [&](int k, icikt_plan* p, const auto& order, int64_t lo, int64_t hi,
                                           WalkTotals& tot, float& d2h_ms) {
    const int r = ensure_edge_buffers(p, p->P);
    return r != ICIKT_OK ? r : edge_walk(p, order, f, lo, hi, p->P, rows[(size_t)k], held, tot, d2h_ms,
                                         adjust ? &parts[(size_t)k] : nullptr);
  });
  if (rc != ICIKT_OK) return rc;
  std::unique_ptr<icikt_edges> res(new (std::nothrow) icikt_edges());
  if (!res) return fail(ICIKT_ERR_ALLOC, "out of host memory");
  res->j_offset = J.y ? (int32_t)J.src.C : 0;
  size_t total = 0;
  for (const auto& r : rows) total += r.size();
  res->rows = std::move(rows[0]);
  try {
    res->rows.reserve(total);
  } catch (const std::bad_alloc&) {
    return fail(ICIKT_ERR_ALLOC, "out of host memory for the selected rows");
  }
  for (size_t k = 1; k < rows.size(); ++k) {
    res->rows.insert(res->rows.end(), rows[k].begin(), rows[k].end());
    std::vector<EdgeRow>().swap(rows[k]);
  }
  float padj_ms = 0.f;
  rc = edge_result(res.get(), f, M, adjust ? [&](icikt_edges* e) { return padj_finish(J, parts, *adjust, e, &padj_ms); }
                                           : std::function<int(icikt_edges*)>());
  if (rc != ICIKT_OK) return rc;
  if (timings) {  // the adjustment's device work counts as epilogue, and the call's device work ends with it
    timings->epilogue_ms += padj_ms;
    timings->total_ms += padj_ms;
  }
  if (max_taumax) *max_taumax = M;
  *out = res.release();
  return ICIKT_OK;
}

int edges_impl(const ColumnSource& s, int64_t n, int64_t C, const double* global_na, int32_t n_global_na,
               const icikt_opts& o, const int32_t* devices, int32_t n_devices, const icikt_edge_filter* filter,
               icikt_edges** out, double* max_taumax, icikt_timings* timings) {
  int rc = check_edge_args(s, n, C, global_na, n_global_na, o, filter, out);
  if (rc == ICIKT_OK) rc = check_window_devices(n_devices);
  if (rc != ICIKT_OK) return rc;
  MultiJob J(n_devices);
  all_pairs_job(J, s, n, global_na, n_global_na, o, devices);
  return edges_run(J, *filter, out, max_taumax, timings);
}

// The one-worker counterpart of topk_merge_block: the worker's lists are the result, copied straight from its plan
// into the arrays of every side; held[r] receives row r's entries, d2h_ms the time of the copy.
int topk_copy_lists(icikt_plan* p, int64_t L, int K, const std::vector<TopkSide>& sides, int32_t* held, float* d2h_ms) {
  std::vector<TopkCol> col;
  try {
    col.resize((size_t)L);
  } catch (const std::bad_alloc&) {
    return fail(ICIKT_ERR_ALLOC, "out of host memory for the lists");
  }
  CK(cudaEventRecord(p->ev[6], p->stream));
  int rc = staged_copy_out(p, col.data(), p->d_tcol.get(), sizeof(TopkCol) * (size_t)L, p->stream);
  const int64_t lk = L * K;
  for (const TopkSide& sd : sides) {
    const int64_t ck = sd.cols * K, at = sd.row0 * K;
    if (rc == ICIKT_OK) rc = staged_copy_out(p, sd.out.index, p->d_tidx.get() + at, sizeof(int32_t) * (size_t)ck, p->stream);
    double* host_field[4] = {sd.raw, sd.out.pvalue, sd.out.taumax, sd.out.completeness};
    for (int f = 0; f < 4 && rc == ICIKT_OK; ++f)
      if (host_field[f])
        rc = staged_copy_out(p, host_field[f], p->d_tlist.get() + f * lk + at, sizeof(double) * (size_t)ck, p->stream);
  }
  if (rc != ICIKT_OK) return rc;
  CK(cudaEventRecord(p->ev[7], p->stream));
  CK(cudaEventSynchronize(p->ev[7]));
  *d2h_ms = ev_ms(p->ev[6], p->ev[7]);
  for (int64_t r = 0; r < L; ++r) held[r] = col[(size_t)r].n;
  return ICIKT_OK;
}

// Worker k's block of list rows [L*k/N, L*(k+1)/N) of the merged lists (L rows: the columns of an all-pairs call,
// the requested sides of a cross call): the merge kernel reads every device's lists in place (J.peer_plan), and the
// block goes straight into the caller's arrays of every side it covers (one block may hold rows of both sides of a
// cross call); held[r] receives row r's entries.  tm: the merge and its copies become d2h_ms.
int topk_merge_block(const MultiJob& J, int k, icikt_plan* p, int64_t L, int K, int by,
                     const std::vector<TopkSide>& sides, int32_t* held, icikt_timings& tm) {
  const int64_t r_lo = L * k / J.n_devices, r_hi = L * (k + 1) / J.n_devices;
  if (r_hi <= r_lo) return ICIKT_OK;
  const size_t blk = (size_t)(r_hi - r_lo) * (size_t)K;
  int rc = ensure_merge_buffers(p, blk);
  if (rc != ICIKT_OK) return rc;
  TopkDeviceMerge m{};
  m.n_dev = J.n_devices;
  for (int j = 0; j < J.n_devices; ++j) {
    m.col[j] = J.peer_plan[(size_t)j]->d_tcol.get();
    m.idx[j] = J.peer_plan[(size_t)j]->d_tidx.get();
    m.list[j] = J.peer_plan[(size_t)j]->d_tlist.get();
  }
  m.C = L;  // the lists' rows: the kernel's columns
  m.c_lo = r_lo;
  m.c_hi = r_hi;
  m.k = K;
  m.by = by;
  m.n = p->d_mn.get();
  m.out_idx = p->d_midx.get();
  m.out = p->d_mlist.get();
  CK(cudaEventRecord(p->ev[6], p->stream));
  const int l = launch_topk_device_merge(m, p->stream);
  if (l < 0) return launch_fail("top-k device merge kernel");
  tm.n_launches += l;
  rc = staged_copy_out(p, held + r_lo, p->d_mn.get(), sizeof(int32_t) * (size_t)(r_hi - r_lo), p->stream);
  for (const TopkSide& sd : sides) {
    const int64_t lo = std::max(r_lo, sd.row0), hi = std::min(r_hi, sd.row0 + sd.cols);
    if (hi <= lo) continue;
    const size_t len = (size_t)(hi - lo) * (size_t)K, from = (size_t)(lo - r_lo) * (size_t)K,
                 to = (size_t)(lo - sd.row0) * (size_t)K;
    if (rc == ICIKT_OK) rc = staged_copy_out(p, sd.out.index + to, p->d_midx.get() + from, sizeof(int32_t) * len, p->stream);
    double* host_field[4] = {sd.raw, sd.out.pvalue, sd.out.taumax, sd.out.completeness};
    for (int f = 0; f < 4 && rc == ICIKT_OK; ++f)
      if (host_field[f])
        rc = staged_copy_out(p, host_field[f] + to, p->d_mlist.get() + f * blk + from, sizeof(double) * len, p->stream);
  }
  if (rc != ICIKT_OK) return rc;
  CK(cudaEventRecord(p->ev[7], p->stream));
  CK(cudaEventSynchronize(p->ev[7]));
  tm.d2h_ms = ev_ms(p->ev[6], p->ev[7]);
  tm.total_ms = ev_ms(p->ev[0], p->ev[7]);
  cudaGetLastError();
  return ICIKT_OK;
}

// The top-k call over the devices of J, its arguments checked: every worker keeps the lists of rows [c_lo, c_hi)
// (columns of the plan) for its slice.  One worker copies its lists out (topk_copy_lists) before its walk is
// finished; several merge a block of rows each into the sides' arrays in a peer phase after it (topk_merge_block).
// Then the host shifts the partners and pads (topk_sides_finish).
int topk_run(MultiJob& J, int K, int by, bool scale, int64_t c_lo, int64_t c_hi, std::vector<TopkSide>& sides,
             double* max_taumax, icikt_timings* timings) {
  int rc = ICIKT_OK;
  for (TopkSide& sd : sides)
    if (rc == ICIKT_OK) rc = topk_raw_buffer(sd.out, sd.cols * K, sd.raw_own, &sd.raw);
  if (rc != ICIKT_OK) return rc;
  const int64_t L = c_hi - c_lo;
  std::vector<int32_t> held;  // without pairs (one column) every list stays empty: padding
  try {
    held.resize((size_t)L);
  } catch (const std::bad_alloc&) {
    return fail(ICIKT_ERR_ALLOC, "out of host memory for the lists");
  }
  double M;
  rc = run_windows(
      J, &M, timings,
      [&](int, icikt_plan* p, const auto& order, int64_t lo, int64_t hi, WalkTotals& tot, float& d2h_ms) {
        int r = ensure_topk_buffers(p, p->P, K, L);
        if (r == ICIKT_OK) r = topk_walk(p, order, c_lo, c_hi, K, by, lo, hi, p->P, tot);
        if (r == ICIKT_OK && J.n_devices == 1) r = topk_copy_lists(p, L, K, sides, held.data(), &d2h_ms);
        return r;
      },
      [&](int k, icikt_plan* p, int r, icikt_timings& tm) {
        return peer_phase(J, k, p, r, "a peer device failed to select its lists", [&] {
          return topk_merge_block(J, k, p, L, K, by, sides, held.data(), tm);
        });
      });
  if (rc != ICIKT_OK) return rc;
  topk_sides_finish(sides, K, [&](int64_t row) { return held[(size_t)row]; }, scale, M);
  if (max_taumax) *max_taumax = M;
  return ICIKT_OK;
}

int topk_impl(const ColumnSource& s, int64_t n, int64_t C, const double* global_na, int32_t n_global_na,
              const icikt_opts& o, const int32_t* devices, int32_t n_devices, int32_t K, int32_t by, int32_t scale_max,
              const TopkOut& out, double* max_taumax, icikt_timings* timings) {
  int rc = check_topk_args(s, n, C, global_na, n_global_na, o, K, by, out.index);
  if (rc == ICIKT_OK) rc = check_window_devices(n_devices);
  if (rc != ICIKT_OK) return rc;
  MultiJob J(n_devices);
  all_pairs_job(J, s, n, global_na, n_global_na, o, devices);
  std::vector<TopkSide> sides{TopkSide{out, 0, C, 0, {}, nullptr}};
  return topk_run(J, K, by, scale_max != 0, 0, C, sides, max_taumax, timings);
}

// ---- the cross calls: the cross order (of the call's range) sliced as above over the Cx + Cy columns of [X | Y]

int cross_pairs_impl(const icikt_input* x, const icikt_input* y, int64_t n, const double* global_na,
                     int32_t n_global_na, const icikt_opts& o, const int32_t* devices, int32_t n_devices, double* raw,
                     double* pvalue, double* taumax, double* completeness, int32_t* status, double* max_taumax,
                     icikt_timings* timings) {
  ColumnSource sx, sy;
  int rc = check_cross_args(x, y, n, global_na, n_global_na, o, true, &sx, &sy);
  if (rc == ICIKT_OK && !raw) rc = fail(ICIKT_ERR_BAD_ARG, "raw is NULL");
  if (rc == ICIKT_OK) rc = check_window_devices(n_devices);
  if (rc != ICIKT_OK) return rc;
  const int64_t first = o.pair_lo, last = (o.pair_hi == 0) ? sx.C * sy.C : o.pair_hi;
  MultiJob J(n_devices);
  cross_job(J, sx, sy, n, global_na, n_global_na, o, devices, first, last);
  double M;
  rc = run_windows(J, &M, timings, [&](int, icikt_plan* p, const auto& order, int64_t lo, int64_t hi,
                                       WalkTotals& tot, float& d2h_ms) {
    const int64_t off = lo - first;
    const int r = ensure_cross_buffers(p);
    return r != ICIKT_OK ? r
                         : cross_pair_walk(p, order, lo, hi, p->P, raw + off, pvalue ? pvalue + off : nullptr,
                                           taumax ? taumax + off : nullptr,
                                           completeness ? completeness + off : nullptr,
                                           status ? status + off : nullptr, tot, d2h_ms);
  });
  if (rc == ICIKT_OK && max_taumax) *max_taumax = M;
  return rc;
}

int cross_edges_impl(const icikt_input* x, const icikt_input* y, int64_t n, const double* global_na,
                     int32_t n_global_na, const icikt_opts& o, const int32_t* devices, int32_t n_devices,
                     const icikt_edge_filter* filter, icikt_edges** out, double* max_taumax, icikt_timings* timings) {
  ColumnSource sx, sy;
  int rc = check_filter_args(filter, out);
  if (rc == ICIKT_OK) rc = check_cross_args(x, y, n, global_na, n_global_na, o, false, &sx, &sy);
  if (rc == ICIKT_OK) rc = check_window_devices(n_devices);
  if (rc != ICIKT_OK) return rc;
  MultiJob J(n_devices);
  cross_job(J, sx, sy, n, global_na, n_global_na, o, devices, 0, sx.C * sy.C);
  return edges_run(J, *filter, out, max_taumax, timings);
}

int cross_topk_impl(const icikt_input* x, const icikt_input* y, int64_t n, const double* global_na,
                    int32_t n_global_na, const icikt_opts& o, const int32_t* devices, int32_t n_devices, int32_t K,
                    int32_t by, int32_t scale_max, const icikt_topk_lists* x_side, const icikt_topk_lists* y_side,
                    double* max_taumax, icikt_timings* timings) {
  int rc = check_k_by(K, by);
  if (rc != ICIKT_OK) return rc;
  if (!x_side && !y_side) return fail(ICIKT_ERR_BAD_ARG, "x_side and y_side are both NULL");
  if ((x_side && !x_side->index) || (y_side && !y_side->index))
    return fail(ICIKT_ERR_BAD_ARG, x_side && !x_side->index ? "x_side->index is NULL" : "y_side->index is NULL");
  ColumnSource sx, sy;
  rc = check_cross_args(x, y, n, global_na, n_global_na, o, false, &sx, &sy);
  if (rc == ICIKT_OK) rc = check_window_devices(n_devices);
  if (rc != ICIKT_OK) return rc;
  MultiJob J(n_devices);
  cross_job(J, sx, sy, n, global_na, n_global_na, o, devices, 0, sx.C * sy.C);
  int64_t c_lo = 0, c_hi = 0;
  std::vector<TopkSide> sides;
  cross_topk_sides(x_side, y_side, sx.C, sy.C, &c_lo, &c_hi, sides);
  return topk_run(J, K, by, scale_max != 0, c_lo, c_hi, sides, max_taumax, timings);
}

// ---- the filtered calls with adjusted p-values (_padj): the all-pairs or cross job of the edges calls, with adjust

int check_padj_method(int32_t method) {
  if (method < ICIKT_PADJ_BONFERRONI || method > ICIKT_PADJ_BY)
    return fail(ICIKT_ERR_BAD_ARG, "method must be one of ICIKT_PADJ_BONFERRONI .. ICIKT_PADJ_BY (Hommel is not offered)");
  return ICIKT_OK;
}

int check_padj(const icikt_padj_filter* a) {
  if (!a) return fail(ICIKT_ERR_BAD_ARG, "adjust is NULL");
  const int rc = check_padj_method(a->method);
  if (rc != ICIKT_OK) return rc;
  if (a->reserved != 0) return fail(ICIKT_ERR_BAD_ARG, "adjust->reserved must be 0");
  return ICIKT_OK;
}

int edges_padj_impl(const icikt_input* x, int64_t n, const double* global_na, int32_t n_global_na, const icikt_opts& o,
                    const int32_t* devices, int32_t n_devices, const icikt_edge_filter* filter,
                    const icikt_padj_filter* adjust, icikt_edges** out, double* max_taumax, icikt_timings* timings) {
  ColumnSource s;
  int rc = check_filter_args(filter, out);
  if (rc == ICIKT_OK) rc = check_padj(adjust);
  if (rc == ICIKT_OK) rc = check_all_pairs_input(x, n, global_na, n_global_na, o, n_devices, &s);
  if (rc != ICIKT_OK) return rc;
  MultiJob J(n_devices);
  all_pairs_job(J, s, n, global_na, n_global_na, o, devices);
  return edges_run(J, *filter, out, max_taumax, timings, adjust);
}

int cross_edges_padj_impl(const icikt_input* x, const icikt_input* y, int64_t n, const double* global_na,
                          int32_t n_global_na, const icikt_opts& o, const int32_t* devices, int32_t n_devices,
                          const icikt_edge_filter* filter, const icikt_padj_filter* adjust, icikt_edges** out,
                          double* max_taumax, icikt_timings* timings) {
  ColumnSource sx, sy;
  int rc = check_filter_args(filter, out);
  if (rc == ICIKT_OK) rc = check_padj(adjust);
  if (rc == ICIKT_OK) rc = check_cross_args(x, y, n, global_na, n_global_na, o, false, &sx, &sy);
  if (rc == ICIKT_OK) rc = check_window_devices(n_devices);
  if (rc != ICIKT_OK) return rc;
  MultiJob J(n_devices);
  cross_job(J, sx, sy, n, global_na, n_global_na, o, devices, 0, sx.C * sy.C);
  return edges_run(J, *filter, out, max_taumax, timings, adjust);
}

// ---- the edge-count calls: the all-pairs or cross job of the filtered calls, with counters instead of rows

// the filters and n_pass of an edge-count call, checked on the host before any device is touched
int check_count_filters(const icikt_edge_filter* filters, int32_t n_filters, const int64_t* n_pass, bool degree,
                        CountSpec* cs) {
  if (n_filters < 1 || n_filters > ICIKT_COUNT_FILTERS_MAX)
    return fail(ICIKT_ERR_BAD_ARG, "n_filters must be in [1, ICIKT_COUNT_FILTERS_MAX]");
  if (!filters) return fail(ICIKT_ERR_BAD_ARG, "filters is NULL");
  if (!n_pass) return fail(ICIKT_ERR_BAD_ARG, "n_pass is NULL");
  for (int32_t f = 0; f < n_filters; ++f) {
    const std::string at = "filter " + std::to_string(f) + ": ";
    if (filters[f].scale_max != 0)
      return fail(ICIKT_ERR_BAD_ARG, at + "scaled thresholds are not counted (scale_max must be 0): count the raw "
                                          "threshold t * max_taumax instead");
    if (filters[f].max_edges != 0) return fail(ICIKT_ERR_BAD_ARG, at + "max_edges must be 0: a count returns no rows");
    if (filters[f].reserved != 0) return fail(ICIKT_ERR_BAD_ARG, at + "reserved must be 0");
    cs->t[f] = filters[f].min_abs_cor;
    cs->a[f] = filters[f].max_pvalue;
  }
  cs->T = n_filters;
  cs->degree = degree;
  return ICIKT_OK;
}

// The counting job over the devices of J, its arguments checked: every worker walks its slice with its own counters,
// and the host sums them into the caller's arrays (integers: the sum is that of one device).  deg: the caller's
// degree tables, each over plan columns [c_lo, c_hi).  With cs.components, comp receives the labels in the same way
// and n_components (may be null) their count: one device's labels as they are, several devices' merged on the host.
int count_run(MultiJob& J, const CountSpec& cs, int64_t* n_pass, const std::vector<DegreeOut>& deg,
              int64_t* status_counts, double* max_taumax, icikt_timings* timings,
              const std::vector<ComponentOut>& comp = {}, int64_t* n_components = nullptr) {
  std::vector<std::vector<unsigned long long>> got((size_t)J.n_devices);  // without pairs every count is 0
  std::vector<std::vector<int32_t>> labels((size_t)J.n_devices);
  double M;
  const int rc = run_windows(J, &M, timings, [&](int k, icikt_plan* p, const auto& order, int64_t lo, int64_t hi,
                                                 WalkTotals& tot, float& d2h_ms) {
    const int r = ensure_walk_buffers(p);
    return r != ICIKT_OK ? r : count_walk(p, order, cs, lo, hi, p->P, tot, got[(size_t)k], labels[(size_t)k], d2h_ms);
  });
  if (rc != ICIKT_OK) return rc;
  const int T = cs.T;
  const int64_t C = J.C;
  auto sum = [&](size_t at) {
    unsigned long long s = 0;
    for (const auto& g : got)
      if (!g.empty()) s += g[at];
    return (int64_t)s;
  };
  for (int f = 0; f < T; ++f) n_pass[f] = sum(16 + (size_t)f);
  if (status_counts)
    for (int c = 0; c < ICIKT_NSTATUS; ++c) status_counts[c] = sum((size_t)c);
  for (const DegreeOut& d : deg)
    if (d.out)
      for (int64_t c = d.c_lo; c < d.c_hi; ++c)
        for (int f = 0; f < T; ++f) d.out[(c - d.c_lo) * T + f] = sum(16 + (size_t)T + (size_t)f * (size_t)C + (size_t)c);
  if (max_taumax) *max_taumax = M;
  if (!cs.components) return ICIKT_OK;
  std::vector<const int32_t*> walked;  // the devices that walked pairs
  const std::vector<unsigned long long>* hooks = nullptr;
  for (size_t k = 0; k < labels.size(); ++k)
    if (!labels[k].empty()) {
      walked.push_back(labels[k].data());
      hooks = &got[k];
    }
  std::vector<int32_t> merged;
  std::vector<int64_t> count((size_t)T);
  const int32_t* lab = walked.empty() ? nullptr : walked[0];
  if (walked.size() == 1) {  // V - hooks: every successful hook joined two trees
    const size_t hooks_at = 16 + (size_t)T + (cs.degree ? (size_t)T * (size_t)C : 0);
    for (int f = 0; f < T; ++f) count[(size_t)f] = C - (int64_t)(*hooks)[hooks_at + (size_t)f];
  } else {  // several slices, or none (no pairs: every vertex alone)
    try {
      merged.resize((size_t)T * (size_t)C);
    } catch (const std::bad_alloc&) {
      return fail(ICIKT_ERR_ALLOC, "out of host memory for the labels");
    }
    merge_component_labels(T, C, walked, merged.data(), count.data());
    lab = merged.data();
  }
  for (const ComponentOut& d : comp)
    if (d.out)
      for (int64_t c = d.c_lo; c < d.c_hi; ++c)
        for (int f = 0; f < T; ++f) d.out[(c - d.c_lo) * T + f] = lab[(size_t)f * (size_t)C + (size_t)c];
  if (n_components) std::copy(count.begin(), count.end(), n_components);
  return ICIKT_OK;
}

// components: the component calls, whose `component` is required (the count calls pass false and nulls)
int count_edges_impl(const icikt_input* x, int64_t n, const double* global_na, int32_t n_global_na, const icikt_opts& o,
                     const int32_t* devices, int32_t n_devices, const icikt_edge_filter* filters, int32_t n_filters,
                     int64_t* n_pass, int64_t* degree, int64_t* status_counts, double* max_taumax,
                     icikt_timings* timings, bool components = false, int32_t* component = nullptr,
                     int64_t* n_components = nullptr) {
  ColumnSource s;
  CountSpec cs;
  int rc = check_count_filters(filters, n_filters, n_pass, degree != nullptr, &cs);
  cs.components = components;
  if (rc == ICIKT_OK && components && !component) rc = fail(ICIKT_ERR_BAD_ARG, "component is NULL");
  if (rc == ICIKT_OK) rc = check_all_pairs_input(x, n, global_na, n_global_na, o, n_devices, &s);
  if (rc != ICIKT_OK) return rc;
  MultiJob J(n_devices);
  all_pairs_job(J, s, n, global_na, n_global_na, o, devices);
  return count_run(J, cs, n_pass, {DegreeOut{degree, 0, s.C}}, status_counts, max_taumax, timings,
                   {ComponentOut{component, 0, s.C}}, n_components);
}

int cross_count_edges_impl(const icikt_input* x, const icikt_input* y, int64_t n, const double* global_na,
                           int32_t n_global_na, const icikt_opts& o, const int32_t* devices, int32_t n_devices,
                           const icikt_edge_filter* filters, int32_t n_filters, int64_t* n_pass, int64_t* x_degree,
                           int64_t* y_degree, int64_t* status_counts, double* max_taumax, icikt_timings* timings,
                           bool components = false, int32_t* x_component = nullptr, int32_t* y_component = nullptr,
                           int64_t* n_components = nullptr) {
  ColumnSource sx, sy;
  CountSpec cs;
  int rc = check_count_filters(filters, n_filters, n_pass, x_degree || y_degree, &cs);
  cs.components = components;
  if (rc == ICIKT_OK && components && !x_component && !y_component)
    rc = fail(ICIKT_ERR_BAD_ARG, "x_component and y_component are both NULL: give at least one");
  if (rc == ICIKT_OK) rc = check_cross_args(x, y, n, global_na, n_global_na, o, false, &sx, &sy);
  if (rc == ICIKT_OK) rc = check_window_devices(n_devices);
  if (rc != ICIKT_OK) return rc;
  MultiJob J(n_devices);
  cross_job(J, sx, sy, n, global_na, n_global_na, o, devices, 0, sx.C * sy.C);
  return count_run(J, cs, n_pass, {DegreeOut{x_degree, 0, sx.C}, DegreeOut{y_degree, sx.C, sx.C + sy.C}},
                   status_counts, max_taumax, timings,
                   {ComponentOut{x_component, 0, sx.C}, ComponentOut{y_component, sx.C, sx.C + sy.C}}, n_components);
}

}  // namespace

extern "C" {

int icikt_all_pairs(const double* data, int64_t n, int64_t C, int64_t ld, const double* global_na,
                    int32_t n_global_na, const icikt_opts* opts, double* raw, double* pvalue,
                    double* taumax, double* completeness, int32_t* status, int64_t* counts,
                    double* max_taumax, icikt_timings* timings) {
  const icikt_opts o = opts_or_default(opts);
  return pairs_impl(dense_source(data, ld, C), n, C, global_na, n_global_na, nullptr, nullptr, 0, o, &o.device, 1,
                    PairArrays{raw, pvalue, taumax, completeness, status, counts}, max_taumax, timings);
}

int icikt_all_pairs_csc(const int64_t* colptr, const int32_t* rowidx, const double* values, int64_t n, int64_t C,
                        const double* global_na, int32_t n_global_na, const icikt_opts* opts, double* raw,
                        double* pvalue, double* taumax, double* completeness, int32_t* status, int64_t* counts,
                        double* max_taumax, icikt_timings* timings) {
  const int rc = check_csc(colptr, rowidx, values, n, C);
  if (rc != ICIKT_OK) return rc;
  const icikt_opts o = opts_or_default(opts);
  return pairs_impl(csc_source(colptr, rowidx, values, C), n, C, global_na, n_global_na, nullptr, nullptr, 0, o,
                    &o.device, 1, PairArrays{raw, pvalue, taumax, completeness, status, counts}, max_taumax, timings);
}

// the options of a _multi call: opts->device, pair_lo and pair_hi are ignored
static icikt_opts multi_opts(const icikt_opts* opts) {
  icikt_opts o = opts_or_default(opts);
  o.pair_lo = o.pair_hi = 0;
  return o;
}

int icikt_all_pairs_multi(const double* data, int64_t n, int64_t C, int64_t ld, const double* global_na,
                          int32_t n_global_na, const icikt_opts* opts, const int32_t* devices,
                          int32_t n_devices, double* raw, double* pvalue, double* taumax,
                          double* completeness, int32_t* status, int64_t* counts, double* max_taumax,
                          icikt_timings* timings) {
  return pairs_impl(dense_source(data, ld, C), n, C, global_na, n_global_na, nullptr, nullptr, 0, multi_opts(opts),
                    devices, n_devices, PairArrays{raw, pvalue, taumax, completeness, status, counts}, max_taumax,
                    timings);
}

int icikt_all_pairs_multi_csc(const int64_t* colptr, const int32_t* rowidx, const double* values, int64_t n,
                              int64_t C, const double* global_na, int32_t n_global_na, const icikt_opts* opts,
                              const int32_t* devices, int32_t n_devices, double* raw, double* pvalue, double* taumax,
                              double* completeness, int32_t* status, int64_t* counts, double* max_taumax,
                              icikt_timings* timings) {
  const int rc = check_csc(colptr, rowidx, values, n, C);
  if (rc != ICIKT_OK) return rc;
  return pairs_impl(csc_source(colptr, rowidx, values, C), n, C, global_na, n_global_na, nullptr, nullptr, 0,
                    multi_opts(opts), devices, n_devices, PairArrays{raw, pvalue, taumax, completeness, status, counts},
                    max_taumax, timings);
}

int icikt_pair_list(const double* data, int64_t n, int64_t C, int64_t ld, const double* global_na,
                    int32_t n_global_na, const int32_t* pi, const int32_t* pj, int64_t P,
                    const icikt_opts* opts, double* raw, double* pvalue, double* taumax,
                    double* completeness, int32_t* status, int64_t* counts, double* max_taumax,
                    icikt_timings* timings) {
  if (!pi || !pj) return fail(ICIKT_ERR_BAD_ARG, "pi and pj must not be NULL");
  const icikt_opts o = opts_or_default(opts);
  return pairs_impl(dense_source(data, ld, C), n, C, global_na, n_global_na, pi, pj, P, o, &o.device, 1,
                    PairArrays{raw, pvalue, taumax, completeness, status, counts}, max_taumax, timings);
}

int icikt_pair_list_csc(const int64_t* colptr, const int32_t* rowidx, const double* values, int64_t n, int64_t C,
                        const double* global_na, int32_t n_global_na, const int32_t* pi, const int32_t* pj, int64_t P,
                        const icikt_opts* opts, double* raw, double* pvalue, double* taumax, double* completeness,
                        int32_t* status, int64_t* counts, double* max_taumax, icikt_timings* timings) {
  if (!pi || !pj) return fail(ICIKT_ERR_BAD_ARG, "pi and pj must not be NULL");
  const int rc = check_csc(colptr, rowidx, values, n, C);
  if (rc != ICIKT_OK) return rc;
  const icikt_opts o = opts_or_default(opts);
  return pairs_impl(csc_source(colptr, rowidx, values, C), n, C, global_na, n_global_na, pi, pj, P, o, &o.device, 1,
                    PairArrays{raw, pvalue, taumax, completeness, status, counts}, max_taumax, timings);
}

// the checks icikt_matrices[_csc] make first
static int check_matrices_one(const ColumnSource& s, const int32_t* pi, const int32_t* pj, const icikt_opts& o) {
  if ((pi == nullptr) != (pj == nullptr)) return fail(ICIKT_ERR_BAD_ARG, "pi and pj must both be given");
  if (!pi && (o.pair_lo != 0 || o.pair_hi != 0))
    return fail(ICIKT_ERR_BAD_ARG, "matrix output needs the whole pair order on one device");
  if (!s.data && !s.csc()) return fail(ICIKT_ERR_BAD_ARG, "data and raw must not be NULL");
  return ICIKT_OK;
}

// ... and icikt_matrices_multi[_csc]
static int check_matrices_multi(const ColumnSource& s, int32_t n_devices) {
  if (!s.data && !s.csc()) return fail(ICIKT_ERR_BAD_ARG, "data must not be NULL");
  return check_window_devices(n_devices);
}

int icikt_matrices(const double* data, int64_t n, int64_t C, int64_t ld, const double* global_na,
                   int32_t n_global_na, const int32_t* pi, const int32_t* pj, int64_t P, const icikt_opts* opts,
                   int32_t scale_max, int32_t diag_good, const int32_t* n_good, double* cor, double* raw,
                   double* pvalue, double* taumax, double* completeness, int64_t* status_counts,
                   double* max_taumax, icikt_timings* timings) {
  const icikt_opts o = opts_or_default(opts);
  const ColumnSource s = dense_source(data, ld, C);
  const int rc = check_matrices_one(s, pi, pj, o);
  if (rc != ICIKT_OK) return rc;
  return matrices_impl(s, n, C, global_na, n_global_na, pi, pj, P, o, &o.device, 1, scale_max, diag_good, n_good, cor,
                       raw, pvalue, taumax, completeness, status_counts, max_taumax, timings);
}

int icikt_matrices_csc(const int64_t* colptr, const int32_t* rowidx, const double* values, int64_t n, int64_t C,
                       const double* global_na, int32_t n_global_na, const int32_t* pi, const int32_t* pj, int64_t P,
                       const icikt_opts* opts, int32_t scale_max, int32_t diag_good, const int32_t* n_good,
                       double* cor, double* raw, double* pvalue, double* taumax, double* completeness,
                       int64_t* status_counts, double* max_taumax, icikt_timings* timings) {
  int rc = check_csc(colptr, rowidx, values, n, C);
  if (rc != ICIKT_OK) return rc;
  const icikt_opts o = opts_or_default(opts);
  const ColumnSource s = csc_source(colptr, rowidx, values, C);
  rc = check_matrices_one(s, pi, pj, o);
  if (rc != ICIKT_OK) return rc;
  return matrices_impl(s, n, C, global_na, n_global_na, pi, pj, P, o, &o.device, 1, scale_max, diag_good, n_good, cor,
                       raw, pvalue, taumax, completeness, status_counts, max_taumax, timings);
}

int icikt_matrices_multi(const double* data, int64_t n, int64_t C, int64_t ld, const double* global_na,
                         int32_t n_global_na, const icikt_opts* opts, const int32_t* devices, int32_t n_devices,
                         int32_t scale_max, int32_t diag_good, const int32_t* n_good, double* cor, double* raw,
                         double* pvalue, double* taumax, double* completeness, int64_t* status_counts,
                         double* max_taumax, icikt_timings* timings) {
  const ColumnSource s = dense_source(data, ld, C);
  const int rc = check_matrices_multi(s, n_devices);
  if (rc != ICIKT_OK) return rc;
  return matrices_impl(s, n, C, global_na, n_global_na, nullptr, nullptr, 0, multi_opts(opts), devices, n_devices,
                       scale_max, diag_good, n_good, cor, raw, pvalue, taumax, completeness, status_counts, max_taumax,
                       timings);
}

int icikt_matrices_multi_csc(const int64_t* colptr, const int32_t* rowidx, const double* values, int64_t n, int64_t C,
                             const double* global_na, int32_t n_global_na, const icikt_opts* opts,
                             const int32_t* devices, int32_t n_devices, int32_t scale_max, int32_t diag_good,
                             const int32_t* n_good, double* cor, double* raw, double* pvalue, double* taumax,
                             double* completeness, int64_t* status_counts, double* max_taumax,
                             icikt_timings* timings) {
  int rc = check_csc(colptr, rowidx, values, n, C);
  if (rc != ICIKT_OK) return rc;
  const ColumnSource s = csc_source(colptr, rowidx, values, C);
  rc = check_matrices_multi(s, n_devices);
  if (rc != ICIKT_OK) return rc;
  return matrices_impl(s, n, C, global_na, n_global_na, nullptr, nullptr, 0, multi_opts(opts), devices, n_devices,
                       scale_max, diag_good, n_good, cor, raw, pvalue, taumax, completeness, status_counts, max_taumax,
                       timings);
}

int icikt_all_pairs_edges(const double* data, int64_t n, int64_t C, int64_t ld, const double* global_na,
                          int32_t n_global_na, const icikt_opts* opts, const icikt_edge_filter* filter,
                          icikt_edges** out, double* max_taumax, icikt_timings* timings) {
  const icikt_opts o = opts_or_default(opts);
  return edges_impl(dense_source(data, ld, C), n, C, global_na, n_global_na, o, &o.device, 1, filter, out, max_taumax,
                    timings);
}

int icikt_all_pairs_edges_csc(const int64_t* colptr, const int32_t* rowidx, const double* values, int64_t n,
                              int64_t C, const double* global_na, int32_t n_global_na, const icikt_opts* opts,
                              const icikt_edge_filter* filter, icikt_edges** out, double* max_taumax,
                              icikt_timings* timings) {
  if (out) *out = nullptr;
  const int rc = check_csc(colptr, rowidx, values, n, C);
  if (rc != ICIKT_OK) return rc;
  const icikt_opts o = opts_or_default(opts);
  return edges_impl(csc_source(colptr, rowidx, values, C), n, C, global_na, n_global_na, o, &o.device, 1, filter, out,
                    max_taumax, timings);
}

int icikt_all_pairs_edges_multi(const double* data, int64_t n, int64_t C, int64_t ld, const double* global_na,
                                int32_t n_global_na, const icikt_opts* opts, const int32_t* devices, int32_t n_devices,
                                const icikt_edge_filter* filter, icikt_edges** out, double* max_taumax,
                                icikt_timings* timings) {
  return edges_impl(dense_source(data, ld, C), n, C, global_na, n_global_na, opts_or_default(opts), devices, n_devices,
                    filter, out, max_taumax, timings);
}

int icikt_all_pairs_edges_multi_csc(const int64_t* colptr, const int32_t* rowidx, const double* values, int64_t n,
                                    int64_t C, const double* global_na, int32_t n_global_na, const icikt_opts* opts,
                                    const int32_t* devices, int32_t n_devices, const icikt_edge_filter* filter,
                                    icikt_edges** out, double* max_taumax, icikt_timings* timings) {
  if (out) *out = nullptr;
  const int rc = check_csc(colptr, rowidx, values, n, C);
  if (rc != ICIKT_OK) return rc;
  return edges_impl(csc_source(colptr, rowidx, values, C), n, C, global_na, n_global_na, opts_or_default(opts), devices,
                    n_devices, filter, out, max_taumax, timings);
}

int icikt_all_pairs_topk(const double* data, int64_t n, int64_t C, int64_t ld, const double* global_na,
                         int32_t n_global_na, const icikt_opts* opts, int32_t k, int32_t by, int32_t scale_max,
                         int32_t* index, int32_t* n_neighbors, double* cor, double* raw, double* pvalue,
                         double* taumax, double* completeness, double* max_taumax, icikt_timings* timings) {
  const icikt_opts o = opts_or_default(opts);
  return topk_impl(dense_source(data, ld, C), n, C, global_na, n_global_na, o, &o.device, 1, k, by, scale_max,
                   TopkOut{index, n_neighbors, cor, raw, pvalue, taumax, completeness}, max_taumax, timings);
}

int icikt_all_pairs_topk_csc(const int64_t* colptr, const int32_t* rowidx, const double* values, int64_t n,
                             int64_t C, const double* global_na, int32_t n_global_na, const icikt_opts* opts,
                             int32_t k, int32_t by, int32_t scale_max, int32_t* index, int32_t* n_neighbors,
                             double* cor, double* raw, double* pvalue, double* taumax, double* completeness,
                             double* max_taumax, icikt_timings* timings) {
  const int rc = check_csc(colptr, rowidx, values, n, C);
  if (rc != ICIKT_OK) return rc;
  const icikt_opts o = opts_or_default(opts);
  return topk_impl(csc_source(colptr, rowidx, values, C), n, C, global_na, n_global_na, o, &o.device, 1, k, by,
                   scale_max, TopkOut{index, n_neighbors, cor, raw, pvalue, taumax, completeness}, max_taumax, timings);
}

int icikt_all_pairs_topk_multi(const double* data, int64_t n, int64_t C, int64_t ld, const double* global_na,
                               int32_t n_global_na, const icikt_opts* opts, const int32_t* devices, int32_t n_devices,
                               int32_t k, int32_t by, int32_t scale_max, int32_t* index, int32_t* n_neighbors,
                               double* cor, double* raw, double* pvalue, double* taumax, double* completeness,
                               double* max_taumax, icikt_timings* timings) {
  return topk_impl(dense_source(data, ld, C), n, C, global_na, n_global_na, opts_or_default(opts), devices, n_devices,
                   k, by, scale_max, TopkOut{index, n_neighbors, cor, raw, pvalue, taumax, completeness}, max_taumax,
                   timings);
}

int icikt_all_pairs_topk_multi_csc(const int64_t* colptr, const int32_t* rowidx, const double* values, int64_t n,
                                   int64_t C, const double* global_na, int32_t n_global_na, const icikt_opts* opts,
                                   const int32_t* devices, int32_t n_devices, int32_t k, int32_t by, int32_t scale_max,
                                   int32_t* index, int32_t* n_neighbors, double* cor, double* raw, double* pvalue,
                                   double* taumax, double* completeness, double* max_taumax, icikt_timings* timings) {
  const int rc = check_csc(colptr, rowidx, values, n, C);
  if (rc != ICIKT_OK) return rc;
  return topk_impl(csc_source(colptr, rowidx, values, C), n, C, global_na, n_global_na, opts_or_default(opts), devices,
                   n_devices, k, by, scale_max, TopkOut{index, n_neighbors, cor, raw, pvalue, taumax, completeness},
                   max_taumax, timings);
}

int icikt_cross_pairs(const icikt_input* x, const icikt_input* y, int64_t n, const double* global_na,
                      int32_t n_global_na, const icikt_opts* opts, double* raw, double* pvalue, double* taumax,
                      double* completeness, int32_t* status, double* max_taumax, icikt_timings* timings) {
  const icikt_opts o = opts_or_default(opts);
  return cross_pairs_impl(x, y, n, global_na, n_global_na, o, &o.device, 1, raw, pvalue, taumax, completeness, status,
                          max_taumax, timings);
}

int icikt_cross_pairs_multi(const icikt_input* x, const icikt_input* y, int64_t n, const double* global_na,
                            int32_t n_global_na, const icikt_opts* opts, const int32_t* devices, int32_t n_devices,
                            double* raw, double* pvalue, double* taumax, double* completeness, int32_t* status,
                            double* max_taumax, icikt_timings* timings) {
  return cross_pairs_impl(x, y, n, global_na, n_global_na, opts_or_default(opts), devices, n_devices, raw, pvalue,
                          taumax, completeness, status, max_taumax, timings);
}

int icikt_cross_edges(const icikt_input* x, const icikt_input* y, int64_t n, const double* global_na,
                      int32_t n_global_na, const icikt_opts* opts, const icikt_edge_filter* filter, icikt_edges** out,
                      double* max_taumax, icikt_timings* timings) {
  const icikt_opts o = opts_or_default(opts);
  return cross_edges_impl(x, y, n, global_na, n_global_na, o, &o.device, 1, filter, out, max_taumax, timings);
}

int icikt_cross_edges_multi(const icikt_input* x, const icikt_input* y, int64_t n, const double* global_na,
                            int32_t n_global_na, const icikt_opts* opts, const int32_t* devices, int32_t n_devices,
                            const icikt_edge_filter* filter, icikt_edges** out, double* max_taumax,
                            icikt_timings* timings) {
  return cross_edges_impl(x, y, n, global_na, n_global_na, opts_or_default(opts), devices, n_devices, filter, out,
                          max_taumax, timings);
}

int icikt_cross_topk(const icikt_input* x, const icikt_input* y, int64_t n, const double* global_na,
                     int32_t n_global_na, const icikt_opts* opts, int32_t k, int32_t by, int32_t scale_max,
                     const icikt_topk_lists* x_side, const icikt_topk_lists* y_side, double* max_taumax,
                     icikt_timings* timings) {
  const icikt_opts o = opts_or_default(opts);
  return cross_topk_impl(x, y, n, global_na, n_global_na, o, &o.device, 1, k, by, scale_max, x_side, y_side,
                         max_taumax, timings);
}

int icikt_cross_topk_multi(const icikt_input* x, const icikt_input* y, int64_t n, const double* global_na,
                           int32_t n_global_na, const icikt_opts* opts, const int32_t* devices, int32_t n_devices,
                           int32_t k, int32_t by, int32_t scale_max, const icikt_topk_lists* x_side,
                           const icikt_topk_lists* y_side, double* max_taumax, icikt_timings* timings) {
  return cross_topk_impl(x, y, n, global_na, n_global_na, opts_or_default(opts), devices, n_devices, k, by, scale_max,
                         x_side, y_side, max_taumax, timings);
}

int icikt_pnorm_device(const double* z, int64_t n, int32_t lower_tail, double* out, int32_t device) {
  if (!z || !out || n < 0) return fail(ICIKT_ERR_BAD_ARG, "bad pnorm arguments");
  int rc = select_device(device);
  if (rc != ICIKT_OK) return rc;
  if (n == 0) return ICIKT_OK;
  DeviceArray<double> dz, dout;
  CK(dz.reserve((size_t)n));
  cudaError_t e = dout.reserve((size_t)n);
  if (e != cudaSuccess) return cuda_fail(e, "cudaMalloc");
  e = cudaMemcpy(dz.get(), z, sizeof(double) * n, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = (launch_pnorm(dz.get(), n, lower_tail, dout.get(), 0) < 0) ? cudaGetLastError() : cudaSuccess;
  if (e == cudaSuccess) e = cudaMemcpy(out, dout.get(), sizeof(double) * n, cudaMemcpyDeviceToHost);
  if (e != cudaSuccess) return cuda_fail(e, "pnorm");
  return ICIKT_OK;
}


int icikt_all_pairs_edges_padj(const icikt_input* x, int64_t n, const double* global_na, int32_t n_global_na,
                               const icikt_opts* opts, const icikt_edge_filter* filter, const icikt_padj_filter* adjust,
                               icikt_edges** out, double* max_taumax, icikt_timings* timings) {
  const icikt_opts o = opts_or_default(opts);
  return edges_padj_impl(x, n, global_na, n_global_na, o, &o.device, 1, filter, adjust, out, max_taumax, timings);
}

int icikt_all_pairs_edges_padj_multi(const icikt_input* x, int64_t n, const double* global_na, int32_t n_global_na,
                                     const icikt_opts* opts, const int32_t* devices, int32_t n_devices,
                                     const icikt_edge_filter* filter, const icikt_padj_filter* adjust, icikt_edges** out,
                                     double* max_taumax, icikt_timings* timings) {
  return edges_padj_impl(x, n, global_na, n_global_na, opts_or_default(opts), devices, n_devices, filter, adjust, out,
                         max_taumax, timings);
}

int icikt_cross_edges_padj(const icikt_input* x, const icikt_input* y, int64_t n, const double* global_na,
                           int32_t n_global_na, const icikt_opts* opts, const icikt_edge_filter* filter,
                           const icikt_padj_filter* adjust, icikt_edges** out, double* max_taumax,
                           icikt_timings* timings) {
  const icikt_opts o = opts_or_default(opts);
  return cross_edges_padj_impl(x, y, n, global_na, n_global_na, o, &o.device, 1, filter, adjust, out, max_taumax,
                               timings);
}

int icikt_cross_edges_padj_multi(const icikt_input* x, const icikt_input* y, int64_t n, const double* global_na,
                                 int32_t n_global_na, const icikt_opts* opts, const int32_t* devices, int32_t n_devices,
                                 const icikt_edge_filter* filter, const icikt_padj_filter* adjust, icikt_edges** out,
                                 double* max_taumax, icikt_timings* timings) {
  return cross_edges_padj_impl(x, y, n, global_na, n_global_na, opts_or_default(opts), devices, n_devices, filter,
                               adjust, out, max_taumax, timings);
}

int icikt_edges_copy_padj(const icikt_edges* e, double* padj) {
  if (!e) return fail(ICIKT_ERR_BAD_ARG, "edges is NULL");
  if (e->n_tests < 0) return fail(ICIKT_ERR_BAD_ARG, "the result holds no adjusted p-values (not from a _padj call)");
  if (!padj && !e->padj.empty()) return fail(ICIKT_ERR_BAD_ARG, "padj is NULL");
  if (!e->padj.empty()) std::memcpy(padj, e->padj.data(), sizeof(double) * e->padj.size());
  return ICIKT_OK;
}

int64_t icikt_edges_n_tests(const icikt_edges* e) { return e ? e->n_tests : -1; }

int icikt_all_pairs_count_edges(const icikt_input* x, int64_t n, const double* global_na, int32_t n_global_na,
                                const icikt_opts* opts, const icikt_edge_filter* filters, int32_t n_filters,
                                int64_t* n_pass, int64_t* degree, int64_t* status_counts, double* max_taumax,
                                icikt_timings* timings) {
  const icikt_opts o = opts_or_default(opts);
  return count_edges_impl(x, n, global_na, n_global_na, o, &o.device, 1, filters, n_filters, n_pass, degree,
                          status_counts, max_taumax, timings);
}

int icikt_all_pairs_count_edges_multi(const icikt_input* x, int64_t n, const double* global_na, int32_t n_global_na,
                                      const icikt_opts* opts, const int32_t* devices, int32_t n_devices,
                                      const icikt_edge_filter* filters, int32_t n_filters, int64_t* n_pass,
                                      int64_t* degree, int64_t* status_counts, double* max_taumax,
                                      icikt_timings* timings) {
  return count_edges_impl(x, n, global_na, n_global_na, opts_or_default(opts), devices, n_devices, filters, n_filters,
                          n_pass, degree, status_counts, max_taumax, timings);
}

int icikt_cross_count_edges(const icikt_input* x, const icikt_input* y, int64_t n, const double* global_na,
                            int32_t n_global_na, const icikt_opts* opts, const icikt_edge_filter* filters,
                            int32_t n_filters, int64_t* n_pass, int64_t* x_degree, int64_t* y_degree,
                            int64_t* status_counts, double* max_taumax, icikt_timings* timings) {
  const icikt_opts o = opts_or_default(opts);
  return cross_count_edges_impl(x, y, n, global_na, n_global_na, o, &o.device, 1, filters, n_filters, n_pass, x_degree,
                                y_degree, status_counts, max_taumax, timings);
}

int icikt_cross_count_edges_multi(const icikt_input* x, const icikt_input* y, int64_t n, const double* global_na,
                                  int32_t n_global_na, const icikt_opts* opts, const int32_t* devices,
                                  int32_t n_devices, const icikt_edge_filter* filters, int32_t n_filters,
                                  int64_t* n_pass, int64_t* x_degree, int64_t* y_degree, int64_t* status_counts,
                                  double* max_taumax, icikt_timings* timings) {
  return cross_count_edges_impl(x, y, n, global_na, n_global_na, opts_or_default(opts), devices, n_devices, filters,
                                n_filters, n_pass, x_degree, y_degree, status_counts, max_taumax, timings);
}

int icikt_all_pairs_components(const icikt_input* x, int64_t n, const double* global_na, int32_t n_global_na,
                               const icikt_opts* opts, const icikt_edge_filter* filters, int32_t n_filters,
                               int64_t* n_pass, int64_t* degree, int32_t* component, int64_t* n_components,
                               int64_t* status_counts, double* max_taumax, icikt_timings* timings) {
  const icikt_opts o = opts_or_default(opts);
  return count_edges_impl(x, n, global_na, n_global_na, o, &o.device, 1, filters, n_filters, n_pass, degree,
                          status_counts, max_taumax, timings, true, component, n_components);
}

int icikt_all_pairs_components_multi(const icikt_input* x, int64_t n, const double* global_na, int32_t n_global_na,
                                     const icikt_opts* opts, const int32_t* devices, int32_t n_devices,
                                     const icikt_edge_filter* filters, int32_t n_filters, int64_t* n_pass,
                                     int64_t* degree, int32_t* component, int64_t* n_components,
                                     int64_t* status_counts, double* max_taumax, icikt_timings* timings) {
  return count_edges_impl(x, n, global_na, n_global_na, opts_or_default(opts), devices, n_devices, filters, n_filters,
                          n_pass, degree, status_counts, max_taumax, timings, true, component, n_components);
}

int icikt_cross_components(const icikt_input* x, const icikt_input* y, int64_t n, const double* global_na,
                           int32_t n_global_na, const icikt_opts* opts, const icikt_edge_filter* filters,
                           int32_t n_filters, int64_t* n_pass, int64_t* x_degree, int64_t* y_degree,
                           int32_t* x_component, int32_t* y_component, int64_t* n_components,
                           int64_t* status_counts, double* max_taumax, icikt_timings* timings) {
  const icikt_opts o = opts_or_default(opts);
  return cross_count_edges_impl(x, y, n, global_na, n_global_na, o, &o.device, 1, filters, n_filters, n_pass, x_degree,
                                y_degree, status_counts, max_taumax, timings, true, x_component, y_component,
                                n_components);
}

int icikt_cross_components_multi(const icikt_input* x, const icikt_input* y, int64_t n, const double* global_na,
                                 int32_t n_global_na, const icikt_opts* opts, const int32_t* devices,
                                 int32_t n_devices, const icikt_edge_filter* filters, int32_t n_filters,
                                 int64_t* n_pass, int64_t* x_degree, int64_t* y_degree, int32_t* x_component,
                                 int32_t* y_component, int64_t* n_components, int64_t* status_counts,
                                 double* max_taumax, icikt_timings* timings) {
  return cross_count_edges_impl(x, y, n, global_na, n_global_na, opts_or_default(opts), devices, n_devices, filters,
                                n_filters, n_pass, x_degree, y_degree, status_counts, max_taumax, timings, true,
                                x_component, y_component, n_components);
}

int icikt_p_adjust(const double* p, int64_t m, int32_t method, int32_t device, double* out, int64_t* n_tests) {
  if (m < 0) return fail(ICIKT_ERR_BAD_ARG, "m must be >= 0");
  if (m > 0 && (!p || !out)) return fail(ICIKT_ERR_BAD_ARG, "p and out must not be NULL");
  int rc = check_padj_method(method);
  if (rc == ICIKT_OK) rc = select_device(device);
  if (rc != ICIKT_OK) return rc;
  int64_t mm = 0;
  if (m > 0) {
    DeviceArray<double> d;
    if (d.reserve(2 * (size_t)m) != cudaSuccess) {
      cudaGetLastError();
      return fail(ICIKT_ERR_ALLOC, "device allocation for " + std::to_string(m) + " p-values failed");
    }
    cudaError_t e = cudaMemcpy(d.get(), p, sizeof(double) * (size_t)m, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = padj_array(d.get(), m, method, d.get() + m, &mm, nullptr, 0);
    if (e == cudaSuccess) e = cudaMemcpy(out, d.get() + m, sizeof(double) * (size_t)m, cudaMemcpyDeviceToHost);
    d.reset();
    if (e != cudaSuccess) {
      cudaGetLastError();
      return e == cudaErrorMemoryAllocation ? fail(ICIKT_ERR_ALLOC, "device allocation for p.adjust failed")
                                            : cuda_fail(e, "p.adjust");
    }
  }
  if (n_tests) *n_tests = mm;
  return ICIKT_OK;
}

}  // extern "C"
