// icikt_internal.h -- host-side declarations shared by the translation units of
// libicikt_b200.so (not part of the public ABI).
#pragma once
#include <cuda_runtime.h>

#include <cstdint>

#include "icikt_common.cuh"

namespace icikt {

// The launchers report failure as a negative count; the CUDA error that caused it is parked here
// (cudaGetLastError clears it) so that the C ABI can put its text into icikt_last_error().
extern thread_local cudaError_t g_launch_error;
extern thread_local const char* g_launch_note;
inline int launch_status(int launches) {
  const cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) return launches;
  g_launch_error = e;
  g_launch_note = "kernel launch";
  return -1;
}
inline int launch_refused(const char* why) {
  g_launch_error = cudaGetLastError();
  g_launch_note = why;
  return -1;
}

// Device-resident per-column tables produced by K1 (layout: DESIGN.md "Data layout in HBM").
struct ColumnTables {
  int64_t n = 0;        // rows (features)
  int64_t C = 0;        // columns (samples)
  int64_t nstride = 0;  // elements per column in the u16 arrays (n rounded up to 64)
  int64_t wstride = 0;  // 32-bit words per column in the bit arrays (n32/32 rounded up to 4)
  uint16_t* perm = nullptr;       // [C][nstride] row ids in ascending value order, missing first
  uint16_t* rank = nullptr;       // [C][nstride] dense rank of every row
  uint16_t* trow = nullptr;       // [C][nstride] rows of tied (non-first-group) elements, sorted order
  uint16_t* trun = nullptr;       // [C][nstride] dense index of their tie group (0..n_tgroups-1), | kLargeFlag
  uint16_t* tend = nullptr;       // [C][nstride] position in sorted order of the tied-row list's entries (rows of small
                                  //              groups; K1 keeps the list index one past the row's group here first)
  uint32_t* tord = nullptr;       // [C][nstride] the tied-row list in walk order: (list index << 16 | rows behind it in its
                                  //              group, 0 for rows of large groups), longest walk first
  uint32_t* nabits = nullptr;     // [C][wstride] bit r: row r missing
  uint32_t* firstbits = nullptr;  // [C][wstride] bit r: row r belongs to the first group (size > 1)
  uint16_t* lgrp = nullptr;       // [C][kLargeStride] (start position, size) of every large tie group
  uint16_t* gstart = nullptr;     // [C][gstride] sorted position where the group of dense rank r starts; [K] = n
  int64_t gstride = 0;            // nstride + 64
  ColStats* stats = nullptr;      // [C]
  int32_t* max_tied = nullptr;    // [4] over the columns: [0] any large tie group, [1] max large groups, [2] max distinct values
};

struct PairRaw {  // what K2 hands to K3
  int64_t dis, ntie, b, g00;
};

struct TiledShape {
  int warps = 0;         // warps per CTA
  int kk = 0;            // 32-element chunks per warp (even)
  int region_bytes = 0;  // ping-pong region per CTA
  int const_region_bytes = 0;  // pass-A buffers of the per-column constant kernel (32 warps)
  int inplace_kk = 0;    // != 0: in-place variant for long vectors (one sequence buffer, kk fixed at compile time)
  bool gmem = false;     // region lives in the global scratch (does not fit shared memory)
  bool const_gmem = false;  // same for the per-column constant kernel
  bool radix = false;    // pass A's levels below the top bits are radix-16 levels (decided by n alone: cconst depends on it)
  int max_ctas = 0;      // CTAs the scratch must provide for
  // filled in by the plan once the scratch exists: bytes per CTA slot and number of slots
  int scratch_stride = 0;
  int scratch_ctas = 0;
};
// tier 0: no column has a large tie group (region = pass A's two u16 buffers, 4*cap bytes);
// tier 1: large tie groups, sorted in place with rank counters in a fifth quarter (5*cap);
// tier 2: so many large groups x distinct values that pass B takes the tied rows instead (8*cap).
// Every tier is enqueued; the launch reads K1's device-side maxima and exits if it is not its turn.
TiledShape tiled_shape(int64_t n, int tier, int64_t wstride, int n_sm, int64_t n_units = 0, bool allow_inplace = true);

struct PairLaunch {
  const ColumnTables* tab;
  const PairUnit* units;  // device
  int64_t n_units;
  const int32_t* pj_list;  // device, may be null
  PairRaw* raw;            // device [P]
  PairComplete* pw = nullptr;  // device [P], complete-observations mode only
  unsigned long long* unit_counter;  // device, zeroed by the launcher
  unsigned char* scratch = nullptr;  // device, global-memory variant only: max_ctas * region_bytes
};

// Scratch of the column kernels (allocated by the plan).
struct ColumnWork {
  unsigned long long* keys_in = nullptr;   // [C][nstride] sort keys by row (long columns only)
  unsigned long long* keys_out = nullptr;  // [C][nstride] keys in sorted order
  uint16_t* vals_in = nullptr;             // [C][nstride] second row-id buffer of the sort, then walk ranks
  uint32_t* gpos = nullptr;                // [C][nstride+64] start position of every tie group
};
bool columns_fused(int64_t n);  // short columns: one kernel per column does everything (and writes tord)

// K1: data (device, column-major, ld) -> tables of columns [col_lo, col_hi).  Does not touch
// tab.max_tied (launch_max_tied derives it from the statistics of all columns).  Returns the
// number of kernel launches or <0.
int launch_columns(const double* d_data, int64_t ld, const double* d_global_na, int n_global_na,
                   int na_inf, ColumnTables& tab, ColumnWork& wk, const TiledShape& sh,
                   unsigned char* scratch, cudaStream_t stream, int64_t col_lo, int64_t col_hi);

// the device-side tier selection of the pair kernel: maxima over the statistics of ALL columns
int launch_max_tied(ColumnTables& tab, cudaStream_t stream);

// pass-A correction constant per column (needs the pair kernel's code path)
int launch_column_consts(ColumnTables& tab, const TiledShape& sh, unsigned char* scratch, cudaStream_t stream,
                         int64_t col_lo, int64_t col_hi);

// K2 (tiled) and K2-naive; both fill raw[P].
// runs only if the device-side maxima written by K1 select `tier`; unit_counter must be zero
int launch_pairs_tiled(const PairLaunch& pl, const TiledShape& sh, int n_sm, int tier, cudaStream_t stream);
int launch_pairs_naive(const PairLaunch& pl, int64_t P, uint32_t* d_scratch, int64_t n_threads,
                       cudaStream_t stream);
size_t naive_scratch_bytes(int64_t n, int64_t n_threads);

// K3: fp64 epilogue, one thread per pair.
struct EpilogueLaunch {
  const ColumnTables* tab;
  const PairUnit* units;
  int64_t n_units;
  int max_unit_pairs = 32;  // longest unit (pairs): sets the threads per unit
  const int32_t* pj_list;
  const PairRaw* raw;
  const PairComplete* pw = nullptr;
  int perspective, alternative, continuity;
  double* tau;
  double* pvalue;
  double* taumax;
  double* completeness;
  int32_t* status;
  int64_t* counts;  // [P][7] or null
  unsigned long long* max_taumax_bits;  // device, initialised to 0 by the launcher's caller
};
int launch_epilogue(const EpilogueLaunch& el, cudaStream_t stream);

// scale_and_reshape on the device (R/kendalltau.R:357-421): symmetric scatter of the per-pair
// results into C x C column-major matrices (any of m[] may be null), cor = raw / max(taumax),
// the diagonal of diag_good; hist[10] counts the pairs of every status class.
struct MatrixFill {
  const PairUnit* units;
  int64_t n_units;
  int max_unit_pairs;
  const int32_t* pj_list;
  const double *tau, *pvalue, *taumax, *completeness;
  const int32_t* status;
  const unsigned long long* max_taumax_bits;
  const ColStats* stats;
  const int32_t* n_good;  // device [C] or null: n - n_na of the column tables
  int64_t n, C;
  int scale_max, diag_good;
  double* m[5];  // cor, raw, pvalue, taumax, completeness
  unsigned long long* hist;  // device [16], zeroed by the caller
};
int launch_matrix_fill(const MatrixFill& mf, cudaStream_t stream);

// The same for a block of columns [c_lo, c_hi) when the pairs were computed on several devices: each
// device fills its block of every matrix from the result arrays of all devices (peer pointers).
constexpr int kMaxMatrixDevices = 16;
struct BlockFill {
  int n_dev;
  const double* tau[kMaxMatrixDevices];
  const double* pvalue[kMaxMatrixDevices];
  const double* taumax[kMaxMatrixDevices];
  const double* completeness[kMaxMatrixDevices];
  const int32_t* status[kMaxMatrixDevices];
  long long pair_lo[kMaxMatrixDevices + 1];  // first pair of every device's slice; [n_dev] = total
  long long n, C, c_lo, c_hi;
  int scale_max, diag_good;
  double max_taumax;       // over all devices; NaN if no pair is valid
  const int32_t* n_good;   // device [C] (diag_good only)
  int best_good;           // max(n_good)
  double* m[5];            // this device's blocks: [c_hi - c_lo][C] each, any may be null
  unsigned long long* hist;  // device [16], zeroed by the caller
};
int launch_matrix_block_fill(const BlockFill& f, cudaStream_t stream);

// pairwise_completeness (R/kendalltau.R:563-629) from missing-row bit masks:
// bits[w][C] (word-major so that neighbouring pairs read neighbouring words)
int launch_missing_bits(const double* d_data, int64_t ld, int64_t n, int64_t C, const double* d_lit, int nlit,
                        int na_nan, int na_inf, uint32_t* bits, int64_t words, cudaStream_t stream);
// pi == null: pair order of icikt_all_pairs with the diagonal appended
int launch_pair_missing(const uint32_t* bits, int64_t words, int64_t n, int64_t C, const int32_t* pi,
                        const int32_t* pj, int64_t P, int32_t* missing, double* completeness,
                        cudaStream_t stream);
int launch_missing_matrix(const uint32_t* bits, int64_t words, int64_t n, int64_t C, double* matrix,
                          cudaStream_t stream);

// CSC input (colptr [C + 1], rowidx / values indexed by the global entry number, rows strictly increasing
// within a column) -> columns [c_lo, c_hi) of the dense column-major n x C matrix `out` (ld = n): stored rows
// get their value, every other row 0.0
int launch_csc_expand(const int64_t* colptr, const int32_t* rowidx, const double* values, int64_t n, int64_t c_lo,
                      int64_t c_hi, double* out, cudaStream_t stream);

// The selection of the filtered all-pairs call (icikt_select.cu): an order-preserving compaction of one window
// of the pair order.  Tiles of kEdgeTile slots: a count pass writes one ballot word per 32 slots and the kept
// rows per tile, one CTA turns the tile counts into exclusive offsets (and `total`), and a scatter pass writes
// the kept slots as EdgeRow (icikt_edges.cuh) in pair order, (i, j) taken from the window's units.
struct EdgeRow;
constexpr int kEdgeTile = 1024;
struct EdgeSelect {
  const PairUnit* units;  // device, the window's units (slots relative to the window)
  int64_t n_units;
  int64_t n_slots;        // pairs in the window
  const double *tau, *pvalue;
  const double *taumax, *completeness;
  const int32_t* status;
  const unsigned long long* max_taumax_bits;  // the maximum so far (K3 of this window has run)
  double min_abs_cor, max_pvalue;             // NaN: no condition
  int scale_max;
  uint32_t* mask;         // device [n_tiles * kEdgeTile / 32]
  uint32_t* tile_offset;  // device [n_tiles]
  unsigned long long* total;  // device, rows kept
  EdgeRow* rows;          // device [n_slots]
};
int launch_edge_select(const EdgeSelect& s, cudaStream_t stream);

// The selection of the top-k all-pairs call (icikt_select.cu), per window: a count pass tests both candidates of
// every valid slot (column i gets partner j, column j gets i) against the column's k-th entry, one CTA scans the
// column counts into bucket offsets, a scatter pass fills the buckets, and one CTA per column merges its bucket
// into the column's sorted list (order of icikt_topk.cuh), gathering the new entries' fields from the window.
// Lists are kept for columns [c_lo, c_hi) only (all columns, or one side of a cross call): a candidate for a column
// outside that range is skipped, and every per-column array is indexed by c - c_lo.
constexpr int kTopkMax = 1024;  // ICIKT_TOPK_MAX
struct TopkCol {
  unsigned long long key;  // the k-th entry's key and partner, once n == k
  int32_t idx;
  int32_t n;               // entries held
};
struct TopkSelect {
  const PairUnit* units;  // device, the window's units (slots relative to the window)
  int64_t n_units;
  int64_t n_slots;        // pairs in the window
  const double *tau, *pvalue, *taumax, *completeness;
  const int32_t* status;
  int64_t c_lo, c_hi;     // the columns that keep lists; L = c_hi - c_lo below
  int k, by;
  uint32_t* col_count;    // device [L]: candidates per column, then the end of every column's bucket
  unsigned long long* total;  // device, candidates in the window
  uint2* cand;            // device [2 n_slots]: (window slot, partner)
  TopkCol* col;           // device [L], zero before the first window
  int32_t* idx;           // device [L k]: the sorted lists
  double *raw, *pv, *tm, *comp;  // device [L k]
};
int launch_topk_select(const TopkSelect& s, cudaStream_t stream);

// The top-k call over several devices (icikt_all_pairs_topk_multi): every device holds the lists of its slice of
// the pair order; one CTA per column of [c_lo, c_hi) folds the devices' lists into one, reading them through peer
// pointers, and gathers the kept entries' fields from the device that holds them.
struct TopkDeviceMerge {
  int n_dev;  // <= kMaxMatrixDevices
  const TopkCol* col[kMaxMatrixDevices];   // [C] each
  const int32_t* idx[kMaxMatrixDevices];   // [C k] each
  const double* list[kMaxMatrixDevices];   // 4 x [C k] each: raw, pvalue, taumax, completeness
  long long C, c_lo, c_hi;
  int k, by;
  int32_t* n;     // this device's block: [c_hi - c_lo] entries kept
  int32_t* out_idx;  // [(c_hi - c_lo) k]
  double* out;    // 4 x [(c_hi - c_lo) k]: raw, pvalue, taumax, completeness
};
int launch_topk_device_merge(const TopkDeviceMerge& m, cudaStream_t stream);

// The counting pass of the edge-count calls (icikt_select.cu), per window: every slot of the window is tested once
// against the T filters (edge_keep_window without scale_max; NaN bounds are no condition), which travel in the launch
// parameters; the counters add up over the windows and nothing else is written.  Degrees are filter-major and indexed
// by the plan's column: entry f * C + c (a cross call's Y column j is the plan's column Cx + j).
constexpr int kCountFiltersMax = 64;  // ICIKT_COUNT_FILTERS_MAX
struct EdgeTally {
  const PairUnit* units;  // device, the window's units (slots relative to the window)
  int64_t n_units;
  int64_t n_slots;        // pairs in the window
  const double *tau, *pvalue;
  const int32_t* status;
  int n_filters;          // T, 1 .. kCountFiltersMax
  int64_t C;              // columns of the plan
  double min_abs_cor[kCountFiltersMax], max_pvalue[kCountFiltersMax];
  unsigned long long* status_counts;  // device [16]: pairs per status class
  unsigned long long* n_pass;         // device [T]
  unsigned long long* degree;         // device [T C], or null
  // The component calls: each filter's union-find forest over the C columns (icikt_components.cuh), filter-major
  // [T][C], and its count of successful hooks [T]; null for the count calls, which then run the kernel without unions.
  int32_t* parent;
  unsigned long long* hooks;
};
int launch_edge_tally(const EdgeTally& s, cudaStream_t stream);
// The forests of the component calls: parent[f C + v] = v before the first window (launch_component_init), every
// entry replaced by its root, the component's smallest vertex, after the last (launch_component_labels).
int launch_component_init(int32_t* parent, int n_filters, int64_t C, cudaStream_t stream);
int launch_component_labels(int32_t* parent, int n_filters, int64_t C, cudaStream_t stream);

// R's p.adjust on the device (icikt_padj.cu, arithmetic in icikt_padj.cuh).  Each returns the first CUDA error.
// counts[0] += the non-NaN values of p[0, n); the keys (padj_key) of those <= bound (NaN: all) are appended at
// keys[counts[1]++], which the caller has made room for.
cudaError_t padj_candidates(const double* p, int64_t n, double bound, unsigned long long* counts,
                            unsigned long long* keys, cudaStream_t stream);
// sorts keys[0, K) (alt: a second buffer of K), then the running max / min of the per-rank values over m tests; on
// return *sorted is the buffer that holds the sorted keys and *vals the other one, holding the scanned values.
// Synchronises the stream.
cudaError_t padj_sort_scan(unsigned long long* keys, unsigned long long* alt, int64_t K, int64_t m, int method,
                           double q, unsigned long long** sorted, double** vals, cudaStream_t stream);
// out[r] = the adjusted value of p[r], every p[r] one of the K sorted keys
cudaError_t padj_lookup(const unsigned long long* sorted, const double* vals, int64_t K, int method, const double* p,
                        int64_t R, double* out, cudaStream_t stream);
// p.adjust(p[0, m), method) into out (device arrays); *n_tests = the non-NaN values; q_ms (may be NULL): the host
// time of BY's sum.  Synchronises the stream.
cudaError_t padj_array(const double* p, int64_t m, int method, double* out, int64_t* n_tests, double* q_ms,
                       cudaStream_t stream);

int launch_pnorm(const double* d_z, int64_t n, int lower, double* d_out, cudaStream_t stream);

int64_t tiled_max_n();

// shared-memory read+write sweep, GB/s for 32-bit and 128-bit accesses (benchmark utility)
int measure_smem_bandwidth(double* gbps32, double* gbps128);
// sustained warp-instruction issue rate (G warp instructions / s over the whole GPU): LOP3 only (ALU
// pipe), IMAD only (FMA pipe), and the two interleaved (benchmark utility)
int measure_issue_rate(double* alu, double* fma, double* mixed);

}  // namespace icikt
