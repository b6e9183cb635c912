/* include/icikt_b200.h -- C ABI of libicikt_b200.so (CUDA, sm_100a).
 *
 * Drop-in boundary for the ONE hot path of ICIKendallTau: the all-pairs / pair-list
 * information-content-informed Kendall-tau-b.  It replaces, in one batched call,
 *
 *   - the R pair loop            R/kendalltau.R:158 + ici_split R/kendalltau.R:280-308
 *     (and kt_split R/kendalltau.R:310-354 for kt_fast),
 *   - the per-pair FFI call      .Call('_ICIKendallTau_ici_kt', ...)  R/RcppExports.R:62-64,
 *                                SEXP _ICIKendallTau_ici_kt(SEXP x6)  src/RcppExports.cpp:83-96,
 *   - the native pair kernel     ici_kt()  src/kendallc.cpp:166-366 and its helpers :5-129,
 *   - the missing-value marking  setup_missing_matrix  R/utils.R:1-23 (fused into the
 *                                per-column preprocessing kernel).
 *
 * (Paths are relative to the reference repository.)  Plain C: pointers and sizes only,
 * no torch / Rcpp types.  There is NO CPU fallback: every entry point returns
 * ICIKT_ERR_NO_DEVICE when no CUDA device is usable.
 *
 * Conventions
 *   data      column-major n x C doubles, leading dimension ld >= n (R matrix layout);
 *             n = features = vector length, C = samples = columns being correlated.
 *   missing   a value is missing if it is NaN/NA, or (na_inf) +-Inf, or equal to one of
 *             the finite literals in global_na[] -- exactly R/utils.R:1-23.  For the
 *             plain ici_kt()/kt_fast() semantics pass n_global_na = 0 and na_inf = 0
 *             (NaN only, src/kendallc.cpp:181,190-191).
 *   pairs     0-based column indices.  icikt_all_pairs enumerates utils::combn(C, 2)
 *             order (0,1),(0,2)...(C-2,C-1) and, if include_diag, appends (0,0)...(C-1,C-1)
 *             exactly as setup_comparisons does when !diag_good (R/kendalltau.R:188-194).
 *   outputs   caller-allocated arrays of length P (pair order above).  Degenerate pairs
 *             get NaN in all four doubles and a non-zero status so the R shim can turn them
 *             into NA_real_ and raise the reference's warnings once per class.
 *   counts    optional int64[P][ICIKT_NCOUNTS]: dis, ntie, xtie, ytie, tot, n_entry, b
 *             (bit-exact against the reference's integer intermediates, for tests).
 */
#ifndef ICIKT_B200_H
#define ICIKT_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ICIKT_ABI_VERSION 1

/* return codes */
#define ICIKT_OK 0
#define ICIKT_ERR_NO_DEVICE (-1)  /* no CUDA device / driver: there is no CPU fallback     */
#define ICIKT_ERR_BAD_ARG (-2)    /* NULL pointer, n < 1, C < 1, bad pair index, ...       */
#define ICIKT_ERR_TOO_LONG (-3)   /* n > icikt_max_n()                                     */
#define ICIKT_ERR_CUDA (-4)       /* CUDA runtime failure, see icikt_last_error()          */
#define ICIKT_ERR_ALLOC (-5)      /* host or device allocation failed                      */
#define ICIKT_ERR_LIMIT (-6)      /* more pairs pass an edge filter than its max_edges     */

/* per-pair status (src/kendallc.cpp line of the matching early return) */
#define ICIKT_STATUS_OK 0
#define ICIKT_STATUS_ALL_NA 1        /* :190-199  silent NA                                 */
#define ICIKT_STATUS_TOO_SHORT 2     /* :224-231  "The vectors only have a single value"     */
#define ICIKT_STATUS_SINGLE_UNIQUE 3 /* :234-244  "... have only a single unique value"      */
#define ICIKT_STATUS_ALL_TIED 4      /* :291-298  "Ties equal the total"                     */
#define ICIKT_STATUS_UNSUPPORTED 9   /* complete-observations mode only, see ICIKT_PERSPECTIVE_COMPLETE */
#define ICIKT_NSTATUS 10             /* length of a per-class count array                    */

#define ICIKT_PERSPECTIVE_GLOBAL 0 /* any string other than "local", src/kendallc.cpp:180 */
#define ICIKT_PERSPECTIVE_LOCAL 1
/* Not an ICI perspective: plain Kendall-tau-b on the rows present in BOTH columns, what
 * kt_fast(use = "pairwise.complete.obs") computes pair by pair (kt_split drops the rows missing
 * in either column and calls ici_kt on the rest, R/kendalltau.R:323-341).  completeness is 1,
 * counts are those of the shared rows; status 9 = a column's missing rows tie with its
 * minimum in fp64 (|min| >= ~1e15), the caller has to filter that pair on the host.          */
#define ICIKT_PERSPECTIVE_COMPLETE 2

#define ICIKT_ALT_TWO_SIDED 0
#define ICIKT_ALT_LESS 1
#define ICIKT_ALT_GREATER 2
#define ICIKT_ALT_OTHER 3 /* unknown string: p-value stays 0, src/kendallc.cpp:323-332 */

#define ICIKT_NCOUNTS 7
#define ICIKT_COUNT_DIS 0
#define ICIKT_COUNT_NTIE 1
#define ICIKT_COUNT_XTIE 2
#define ICIKT_COUNT_YTIE 3
#define ICIKT_COUNT_TOT 4
#define ICIKT_COUNT_N_ENTRY 5
#define ICIKT_COUNT_B 6 /* rows missing in both columns */

#define ICIKT_KERNEL_TILED 0 /* one CTA per pair, shared-memory bit-partition counting */
#define ICIKT_KERNEL_NAIVE 1 /* one thread per pair, Fenwick tree in global memory
                                (the internal baseline BASELINE.json names)           */

typedef struct icikt_opts {
  int32_t perspective;  /* ICIKT_PERSPECTIVE_*  (ici_kt argument `perspective`)          */
  int32_t alternative;  /* ICIKT_ALT_*          (ici_kt argument `alternative`)          */
  int32_t continuity;   /* 0/1                  (ici_kt argument `continuity`)           */
  int32_t include_diag; /* all-pairs only: append the C (i,i) pairs (!diag_good)         */
  int32_t na_inf;       /* treat +-Inf as missing (Inf present in global_na)             */
  int32_t device;       /* CUDA device ordinal to run on                                 */
  int32_t kernel;       /* ICIKT_KERNEL_*                                                */
  int32_t want_counts;  /* plan API: allocate and fill the int64 counts (one-shot: set from `counts`) */
  int64_t pair_lo;      /* compute only pairs [pair_lo, pair_hi) of the pair order; the   */
  int64_t pair_hi;      /* output arrays are still indexed from 0 = pair_lo.  0,0 = all.  */
} icikt_opts;

/* A pipelined one-shot call (see icikt_stage_table) overlaps the copies with the kernels: columns_ms,
 * pairs_ms and epilogue_ms are then sums over its launches, h2d_ms runs from the start of the call until
 * the last column has landed, d2h_ms from the first result copy to the last, and the parts exceed total_ms. */
typedef struct icikt_timings { /* milliseconds, CUDA events on the library's streams */
  float h2d_ms;      /* host -> device copy of the data matrix (CSC input: of its arrays) */
  float columns_ms;  /* per-column preprocessing kernels (K1; CSC input: with the expansion) */
  float pairs_ms;    /* pair kernel (K2) alone                                        */
  float epilogue_ms; /* fp64 epilogue kernel (K3)                                     */
  float d2h_ms;      /* device -> host copy of the results                            */
  float total_ms;    /* first to last event                                           */
  int32_t n_launches; /* kernels launched by the last columns + pairs calls           */
  int32_t reserved;
} icikt_timings;

/* defaults: global, two.sided, no continuity, no diag, NaN-only missing, device 0, tiled */
void icikt_default_opts(icikt_opts* o);

int icikt_abi_version(void);
int icikt_device_count(void);          /* 0 when no usable device                      */
int64_t icikt_max_n(void);             /* longest supported vector (features)          */
const char* icikt_last_error(void);    /* thread-local message of the last failure     */

/* Replaces R/kendalltau.R:158 for the all-pairs case.  P = C*(C-1)/2 (+ C).
 * pvalue/taumax/completeness/status/counts/max_taumax/timings may be NULL.
 * max_taumax receives max(taumax, na.rm = TRUE) over the computed pairs
 * (R/kendalltau.R:368-370), or NaN if every pair is degenerate.                      */
int icikt_all_pairs(const double* data, int64_t n, int64_t C, int64_t ld,
                    const double* global_na, int32_t n_global_na, const icikt_opts* opts,
                    double* raw, double* pvalue, double* taumax, double* completeness,
                    int32_t* status, int64_t* counts, double* max_taumax,
                    icikt_timings* timings);

/* The same over several GPUs of one box in ONE call (what `computation$ncore` workers are to the
 * reference, R/kendalltau.R:250-253): device k of devices[0..n_devices) preprocesses all columns
 * and computes the k-th contiguous slice of the pair order straight into the caller's arrays;
 * max_taumax is the maximum over the devices.  No collective is involved: pairs are independent
 * (SURVEY.md 8e).  devices == NULL means ordinals 0..n_devices-1; opts->device, pair_lo and
 * pair_hi are ignored.  timings (may be NULL) receives the slowest device's figures.
 * With n_devices == 1 the work runs on the calling thread, whose current CUDA device is devices[0]
 * afterwards, as after every single-device call, and it is icikt_all_pairs' work: a large input takes
 * the pipelined path (icikt_stage_table), with the timings described above icikt_timings.      */
int icikt_all_pairs_multi(const double* data, int64_t n, int64_t C, int64_t ld,
                          const double* global_na, int32_t n_global_na, const icikt_opts* opts,
                          const int32_t* devices, int32_t n_devices, double* raw, double* pvalue,
                          double* taumax, double* completeness, int32_t* status, int64_t* counts,
                          double* max_taumax, icikt_timings* timings);

/* Same for an explicit pair list (include_only, ici_kt(x, y) with C = 2 and P = 1,
 * kt_fast incl. (i,i) pairs).  pi[k], pj[k] in [0, C).                               */
int icikt_pair_list(const double* data, int64_t n, int64_t C, int64_t ld,
                    const double* global_na, int32_t n_global_na, const int32_t* pi,
                    const int32_t* pj, int64_t P, const icikt_opts* opts, double* raw,
                    double* pvalue, double* taumax, double* completeness, int32_t* status,
                    int64_t* counts, double* max_taumax, icikt_timings* timings);

/* ici_kendalltau(return_matrix = TRUE) in one call: icikt_all_pairs (pi == NULL; the diagonal
 * pairs are computed iff !diag_good, like setup_comparisons) or icikt_pair_list (pi, pj, P)
 * followed by icikt_plan_download_matrices; see there for the outputs.                      */
int icikt_matrices(const double* data, int64_t n, int64_t C, int64_t ld, const double* global_na,
                   int32_t n_global_na, const int32_t* pi, const int32_t* pj, int64_t P,
                   const icikt_opts* opts, int32_t scale_max, int32_t diag_good,
                   const int32_t* n_good, double* cor, double* raw, double* pvalue, double* taumax,
                   double* completeness, int64_t* status_counts, double* max_taumax,
                   icikt_timings* timings);

/* icikt_matrices (all pairs) over several GPUs of one box in ONE call: the pair order is sliced over
 * the devices like icikt_all_pairs_multi (sharded K1 + peer gather of the tables), then device k
 * fills columns [C*k/N, C*(k+1)/N) of the five matrices -- reading the per-pair results of the other
 * devices in place over NVLink -- and copies its block straight into the caller's arrays, so the
 * 5 x C x C doubles leave over N PCIe links at once.  Needs peer access between the devices; without
 * it (or with one device) the call runs icikt_matrices on devices[0].  n_devices <= 16.          */
int icikt_matrices_multi(const double* data, int64_t n, int64_t C, int64_t ld, const double* global_na,
                         int32_t n_global_na, const icikt_opts* opts, const int32_t* devices,
                         int32_t n_devices, int32_t scale_max, int32_t diag_good, const int32_t* n_good,
                         double* cor, double* raw, double* pvalue, double* taumax, double* completeness,
                         int64_t* status_counts, double* max_taumax, icikt_timings* timings);

/* pairwise_completeness (R/kendalltau.R:563-629): missing[k] = rows missing in column pi[k] or
 * pj[k] (missing_either, :626-629), completeness[k] = 1 - missing/n (:617).  Here, as in
 * setup_missing_matrix (R/utils.R:1-23), NaN/NA rows are missing only if global_na holds a NaN,
 * +-Inf rows only if it holds an Inf.  pi == pj == NULL: all pairs in combn order followed by
 * the C diagonal pairs (diag_good = FALSE, :586), P = C*(C-1)/2 + C outputs; then `matrix`
 * (C x C, may be NULL) receives the symmetric completeness matrix (:598-605).  missing and
 * completeness may be NULL.  No pair kernel runs: bit masks and popc only.                  */
int icikt_pairwise_completeness(const double* data, int64_t n, int64_t C, int64_t ld,
                                const double* global_na, int32_t n_global_na, int32_t device,
                                const int32_t* pi, const int32_t* pj, int64_t P, int32_t* missing,
                                double* completeness, double* matrix);

/* ---- sparse (CSC) input: the six calls above with (data, n, C, ld) replaced by a compressed sparse
 * column matrix (colptr, rowidx, values, n, C), the layout of scipy.sparse.csc_matrix, AnnData's X and R's
 * dgCMatrix: the stored entries of column c are rows rowidx[colptr[c] .. colptr[c+1]) with values[] at the
 * same positions; colptr has C + 1 entries, colptr[0] = 0, colptr[C] = nnz.  Within a column the rows must
 * lie in [0, n) and strictly increase (sorted, no duplicates).  An entry that is not stored is the value
 * 0.0, and every value -- stored or not -- then goes through the usual missing-value rules: with the
 * default global_na = c(NA, Inf, 0) the stored entries are exactly the present values.  Each result is
 * bit for bit the dense call's on the expanded matrix.  The arrays are checked on the host before any
 * device work (ICIKT_ERR_BAD_ARG naming the column).  Only the stored entries travel to the device, where
 * a kernel rebuilds the dense columns ahead of the per-column preprocessing; in `timings`, h2d_ms covers
 * the copies of the CSC arrays and columns_ms includes that expansion.                                 */
int icikt_all_pairs_csc(const int64_t* colptr, const int32_t* rowidx, const double* values, int64_t n,
                        int64_t C, const double* global_na, int32_t n_global_na, const icikt_opts* opts,
                        double* raw, double* pvalue, double* taumax, double* completeness, int32_t* status,
                        int64_t* counts, double* max_taumax, icikt_timings* timings);
int icikt_all_pairs_multi_csc(const int64_t* colptr, const int32_t* rowidx, const double* values, int64_t n,
                              int64_t C, const double* global_na, int32_t n_global_na,
                              const icikt_opts* opts, const int32_t* devices, int32_t n_devices,
                              double* raw, double* pvalue, double* taumax, double* completeness,
                              int32_t* status, int64_t* counts, double* max_taumax,
                              icikt_timings* timings);
int icikt_pair_list_csc(const int64_t* colptr, const int32_t* rowidx, const double* values, int64_t n,
                        int64_t C, const double* global_na, int32_t n_global_na, const int32_t* pi,
                        const int32_t* pj, int64_t P, const icikt_opts* opts, double* raw,
                        double* pvalue, double* taumax, double* completeness, int32_t* status,
                        int64_t* counts, double* max_taumax, icikt_timings* timings);
int icikt_matrices_csc(const int64_t* colptr, const int32_t* rowidx, const double* values, int64_t n,
                       int64_t C, const double* global_na, int32_t n_global_na, const int32_t* pi,
                       const int32_t* pj, int64_t P, const icikt_opts* opts, int32_t scale_max,
                       int32_t diag_good, const int32_t* n_good, double* cor, double* raw,
                       double* pvalue, double* taumax, double* completeness, int64_t* status_counts,
                       double* max_taumax, icikt_timings* timings);
int icikt_matrices_multi_csc(const int64_t* colptr, const int32_t* rowidx, const double* values,
                             int64_t n, int64_t C, const double* global_na, int32_t n_global_na,
                             const icikt_opts* opts, const int32_t* devices, int32_t n_devices,
                             int32_t scale_max, int32_t diag_good, const int32_t* n_good, double* cor,
                             double* raw, double* pvalue, double* taumax, double* completeness,
                             int64_t* status_counts, double* max_taumax, icikt_timings* timings);
int icikt_pairwise_completeness_csc(const int64_t* colptr, const int32_t* rowidx, const double* values,
                                    int64_t n, int64_t C, const double* global_na,
                                    int32_t n_global_na, int32_t device, const int32_t* pi,
                                    const int32_t* pj, int64_t P, int32_t* missing,
                                    double* completeness, double* matrix);

/* ---- all pairs, filtered on the device: only the pairs that pass a correlation or p-value threshold (the
 * network of a wide matrix) come back, as a long table in host memory owned by the library.  Device memory
 * does not depend on the number of pairs P: it is the per-column tables plus one window of W pairs of the
 * pair order (ICIKT_EDGE_WINDOW, default 2^26), which is computed, filtered and copied out while the next
 * window runs.  A pair is an edge iff
 *
 *   status == 0  &&  (isnan(min_abs_cor) || fabs(cor) >= min_abs_cor)  &&  (isnan(max_pvalue) || pvalue <= max_pvalue)
 *
 * with cor = scale_max ? raw / M : raw, M = max(taumax) over ALL computed pairs (the IEEE division of
 * icikt_plan_download_matrices).  A NaN bound is no condition.  Edges are in the pair order of icikt_all_pairs
 * (combn order, then the diagonal if include_diag), and every field is bit for bit what icikt_all_pairs
 * returns for that pair: the result is the full per-pair result, masked.
 * Options: perspective global or local, alternative, continuity, na_inf, device, include_diag.  Refused with
 * ICIKT_ERR_BAD_ARG before any device is touched: pair_lo / pair_hi != 0, ICIKT_PERSPECTIVE_COMPLETE,
 * ICIKT_KERNEL_NAIVE, want_counts, max_edges < 0, a NULL filter or out.  max_edges > 0 fails the call with
 * ICIKT_ERR_LIMIT once more rows than that are held; with scale_max that count is taken after each window
 * against the maximum so far, so it may include rows the final maximum removes.  On success *out receives
 * the rows (free with icikt_edges_free), max_taumax (may be NULL) M or NaN.  timings (may be NULL): pairs_ms
 * is the sum of K2 over the windows, epilogue_ms of K3 and the selection, h2d_ms / d2h_ms cover their copies. */
typedef struct icikt_edge_filter {
  double min_abs_cor; /* NaN: no condition on cor                                     */
  double max_pvalue;  /* NaN: no condition on the p-value                             */
  int32_t scale_max;  /* cor = raw / max(taumax) over all pairs, or raw               */
  int32_t reserved;   /* 0                                                            */
  int64_t max_edges;  /* 0: no limit; otherwise fail with ICIKT_ERR_LIMIT             */
} icikt_edge_filter;

typedef struct icikt_edges icikt_edges; /* result rows in host memory owned by the library */

int icikt_all_pairs_edges(const double* data, int64_t n, int64_t C, int64_t ld, const double* global_na,
                          int32_t n_global_na, const icikt_opts* opts, const icikt_edge_filter* filter,
                          icikt_edges** out, double* max_taumax, icikt_timings* timings);
/* the same for a CSC matrix (see the sparse calls above) */
int icikt_all_pairs_edges_csc(const int64_t* colptr, const int32_t* rowidx, const double* values, int64_t n,
                              int64_t C, const double* global_na, int32_t n_global_na, const icikt_opts* opts,
                              const icikt_edge_filter* filter, icikt_edges** out, double* max_taumax,
                              icikt_timings* timings);
/* number of rows (0 for NULL) */
int64_t icikt_edges_count(const icikt_edges* e);
/* the rows into caller arrays of icikt_edges_count(e) entries; any pointer may be NULL; cor as defined above.
 * All-pairs result: i < j, or i == j for the diagonal pairs.  Cross result (icikt_cross_edges): i in [0, Cx) is
 * X's column and j in [0, Cy) is Y's own column index. */
int icikt_edges_copy(const icikt_edges* e, int32_t* i, int32_t* j, double* cor, double* raw, double* pvalue,
                     double* taumax, double* completeness);
void icikt_edges_free(icikt_edges* e);

/* ---- all pairs, each column's k most correlated partners (the kNN table of a wide matrix), selected on the
 * device over the same windows of the pair order as the filtered call above (ICIKT_EDGE_WINDOW).  For column c
 * the candidates are every d != c whose pair (min(c, d), max(c, d)) has status == 0; degenerate pairs are never
 * candidates and raise no warning.  Candidates are ranked by a strict total order:
 *
 *   by = ICIKT_TOPK_ABS:    |raw| descending, then d ascending
 *   by = ICIKT_TOPK_SIGNED:  raw  descending, then d ascending  (-0.0 equal to +0.0)
 *
 * and column c keeps the first min(k, #candidates) of them, best first.  The ranking is on raw, not on cor:
 * two raws that differ keep their order even where they round to the same cor = raw / M.
 * Outputs are caller-allocated C x k arrays, entry r of column c at c*k + r: index (required) the partner d;
 * cor (scale_max ? raw / M : raw, M = max(taumax) over all computed pairs, the IEEE division of
 * icikt_plan_download_matrices), raw, pvalue, taumax, completeness (each may be NULL) bit for bit what
 * icikt_all_pairs returns for that pair.  Unused entries hold index -1 and a quiet NaN in every double;
 * n_neighbors [C] (may be NULL) the entries kept.  k > C - 1 only pads; C == 1 pads everything and M is NaN.
 * Device memory does not depend on P: the per-column tables, one window of pairs, its candidates (16 B per
 * pair) and the lists (36 B per entry).
 * Options: perspective global or local, alternative, continuity, na_inf, device.  Refused with
 * ICIKT_ERR_BAD_ARG before any device is touched: k < 1 or k > ICIKT_TOPK_MAX, by not ABS or SIGNED, a NULL
 * index, include_diag, pair_lo / pair_hi != 0, ICIKT_PERSPECTIVE_COMPLETE, ICIKT_KERNEL_NAIVE, want_counts.
 * max_taumax (may be NULL) M or NaN.  timings (may be NULL): pairs_ms is the sum of K2 over the windows,
 * epilogue_ms of K3 and the selection, d2h_ms the copy of the lists. */
#define ICIKT_TOPK_ABS 0
#define ICIKT_TOPK_SIGNED 1
#define ICIKT_TOPK_MAX 1024

int icikt_all_pairs_topk(const double* data, int64_t n, int64_t C, int64_t ld, const double* global_na,
                         int32_t n_global_na, const icikt_opts* opts, int32_t k, int32_t by, int32_t scale_max,
                         int32_t* index, int32_t* n_neighbors, double* cor, double* raw, double* pvalue,
                         double* taumax, double* completeness, double* max_taumax, icikt_timings* timings);
/* the same for a CSC matrix (see the sparse calls above) */
int icikt_all_pairs_topk_csc(const int64_t* colptr, const int32_t* rowidx, const double* values, int64_t n,
                             int64_t C, const double* global_na, int32_t n_global_na, const icikt_opts* opts,
                             int32_t k, int32_t by, int32_t scale_max, int32_t* index, int32_t* n_neighbors,
                             double* cor, double* raw, double* pvalue, double* taumax, double* completeness,
                             double* max_taumax, icikt_timings* timings);

/* ---- the filtered and the top-k all-pairs calls over several GPUs of one box in ONE call.  The pair order is sliced
 * over the devices as in icikt_all_pairs_multi (sharded K1 + peer gather of the tables when every pair of devices has
 * peer access, otherwise every device preprocesses all columns), and device k walks its slice in windows of
 * min(ICIKT_EDGE_WINDOW, slice) pairs.  Edges: every device keeps the rows of its slice against its own running
 * maximum (a superset of the final rows); the host trims them with the final maximum M over all devices and joins
 * them in slice order.  Top-k: every device keeps the lists of its slice; then device k merges the lists of all
 * devices for columns [C*k/N, C*(k+1)/N), reading them in place through peer access, and copies its block straight
 * into the caller's arrays.  Without peer access between distinct devices, or with one device, the top-k call runs
 * icikt_all_pairs_topk on devices[0]; the edges call runs icikt_all_pairs_edges there with one device.
 *
 *   - Same result as one device: every output (rows, their order and fields, cor, max_taumax, index, n_neighbors,
 *     the padding, what icikt_edges_copy returns) is bit for bit that of the single-device call.
 *   - devices == NULL means ordinals 0..n_devices-1; repeated ordinals are allowed; 1 <= n_devices <= 16.
 *     opts->device is ignored.
 *   - Refused with ICIKT_ERR_BAD_ARG before any device is touched: whatever the single-device call refuses, and
 *     n_devices out of range.
 *   - max_edges counts the rows held over all devices.  Without scale_max or without min_abs_cor the call fails with
 *     ICIKT_ERR_LIMIT exactly when more than max_edges pairs pass; with both, the held count may include rows the
 *     final maximum removes, as in the single-device call.  When one device crosses the limit, the others stop at
 *     their next window boundary.
 *   - timings (may be NULL): the slowest device's figures, n_launches summed over the devices; for top-k, d2h_ms is
 *     the merge of the device's block with its copy out. */
int icikt_all_pairs_edges_multi(const double* data, int64_t n, int64_t C, int64_t ld, const double* global_na,
                                int32_t n_global_na, const icikt_opts* opts, const int32_t* devices, int32_t n_devices,
                                const icikt_edge_filter* filter, icikt_edges** out, double* max_taumax,
                                icikt_timings* timings);
int icikt_all_pairs_edges_multi_csc(const int64_t* colptr, const int32_t* rowidx, const double* values, int64_t n,
                                    int64_t C, const double* global_na, int32_t n_global_na, const icikt_opts* opts,
                                    const int32_t* devices, int32_t n_devices, const icikt_edge_filter* filter,
                                    icikt_edges** out, double* max_taumax, icikt_timings* timings);
int icikt_all_pairs_topk_multi(const double* data, int64_t n, int64_t C, int64_t ld, const double* global_na,
                               int32_t n_global_na, const icikt_opts* opts, const int32_t* devices, int32_t n_devices,
                               int32_t k, int32_t by, int32_t scale_max, int32_t* index, int32_t* n_neighbors,
                               double* cor, double* raw, double* pvalue, double* taumax, double* completeness,
                               double* max_taumax, icikt_timings* timings);
int icikt_all_pairs_topk_multi_csc(const int64_t* colptr, const int32_t* rowidx, const double* values, int64_t n,
                                   int64_t C, const double* global_na, int32_t n_global_na, const icikt_opts* opts,
                                   const int32_t* devices, int32_t n_devices, int32_t k, int32_t by, int32_t scale_max,
                                   int32_t* index, int32_t* n_neighbors, double* cor, double* raw, double* pvalue,
                                   double* taumax, double* completeness, double* max_taumax, icikt_timings* timings);

/* ---- cross calls: every column of a matrix X (n x Cx) against every column of a matrix Y (n x Cy) with the same n
 * rows -- query samples against a reference panel, two batches, two feature sets measured on the same samples.
 *
 *   - Pair order: x-major, pair p = i * Cy + j is (x column i, y column j), so a per-pair array of the whole order is
 *     the Cx x Cy matrix in row-major order.
 *   - Exactness: X's column is the reference's `x` (first column).  Every field is bit for bit what icikt_pair_list
 *     returns on the dense [X | Y] (ld = n) with pi = i and pj = Cx + j, and max_taumax is the maximum over the
 *     computed pairs.  The per-column statistics of K1 depend on the column alone, so preprocessing [X | Y] gives
 *     every column the tables it gets in that call.
 *   - Input: each matrix is an icikt_input, dense or CSC (see the sparse calls above; CSC arrays are checked before
 *     any device work, and a message names the matrix, x or y, and the column).
 *   - Options: perspective global or local, alternative, continuity, na_inf, device, and (icikt_cross_pairs only)
 *     pair_lo / pair_hi.  Refused with ICIKT_ERR_BAD_ARG before any device is touched: x or y NULL, a descriptor
 *     with both forms or neither, C < 1, n < 1, ld < n, Cx + Cy > INT32_MAX, bad CSC, include_diag,
 *     ICIKT_PERSPECTIVE_COMPLETE, ICIKT_KERNEL_NAIVE, want_counts, pair_lo / pair_hi outside [0, Cx * Cy] (non-zero
 *     on the edges and top-k calls), and whatever icikt_all_pairs_edges / icikt_all_pairs_topk refuse of their own
 *     arguments.  A well-formed call without a device returns ICIKT_ERR_NO_DEVICE.
 *   - Device memory does not depend on the number of pairs: all three calls walk the cross order in windows of
 *     ICIKT_EDGE_WINDOW pairs, as the filtered all-pairs calls do.  timings as there. */
typedef struct icikt_input {
  int64_t C;                 /* columns                                                   */
  const double* data;        /* dense column-major, ld >= n; NULL for CSC                 */
  int64_t ld;
  const int64_t* colptr;     /* CSC as in the *_csc calls (C + 1 entries); NULL for dense */
  const int32_t* rowidx;
  const double* values;
} icikt_input;

/* Per-pair results of pairs [pair_lo, pair_hi) of the cross order (0, 0: all Cx * Cy), straight into caller arrays
 * indexed from 0 = pair_lo.  pvalue / taumax / completeness / status / max_taumax / timings may be NULL, raw may not.
 * Each window's results are copied to the caller while the next window is computed. */
int icikt_cross_pairs(const icikt_input* x, const icikt_input* y, int64_t n, const double* global_na,
                      int32_t n_global_na, const icikt_opts* opts, double* raw, double* pvalue, double* taumax,
                      double* completeness, int32_t* status, double* max_taumax, icikt_timings* timings);

/* The filtered call (icikt_all_pairs_edges) on the cross order: the same filter, predicate, prefilter, final trim
 * with M and max_edges.  Rows are in cross order; icikt_edges_copy gives i as X's and j as Y's column index. */
int icikt_cross_edges(const icikt_input* x, const icikt_input* y, int64_t n, const double* global_na,
                      int32_t n_global_na, const icikt_opts* opts, const icikt_edge_filter* filter, icikt_edges** out,
                      double* max_taumax, icikt_timings* timings);

/* Each column's k best partners in the OTHER matrix, in the order of icikt_all_pairs_topk (|raw| or raw descending,
 * then partner ascending; degenerate pairs are never candidates).  x_side receives Cx x k lists whose partners are Y
 * indices, y_side Cy x k lists whose partners are X indices; entry r of column c at c * k + r, padding index -1 and a
 * quiet NaN, k > the other side's width only pads.  Either side may be NULL, not both; a given side needs index, its
 * other pointers may be NULL.  Lists are held on the device for the requested sides only: 36 B x k x their columns. */
typedef struct icikt_topk_lists {
  int32_t* index;        /* [C k] partner, -1 where unused      */
  int32_t* n_neighbors;  /* [C] entries kept                    */
  double* cor;           /* [C k] each, NaN where unused        */
  double* raw;
  double* pvalue;
  double* taumax;
  double* completeness;
} icikt_topk_lists;

int icikt_cross_topk(const icikt_input* x, const icikt_input* y, int64_t n, const double* global_na,
                     int32_t n_global_na, const icikt_opts* opts, int32_t k, int32_t by, int32_t scale_max,
                     const icikt_topk_lists* x_side, const icikt_topk_lists* y_side, double* max_taumax,
                     icikt_timings* timings);

/* ---- the cross calls over several GPUs of one box in ONE call, as the filtered all-pairs multi calls above.  The
 * cross order (of [pair_lo, pair_hi) for icikt_cross_pairs_multi) is sliced over the devices, and device k walks its
 * slice in windows of min(ICIKT_EDGE_WINDOW, slice) pairs.  The columns are prepared as in icikt_all_pairs_multi
 * over the Cx + Cy columns of [X | Y]: sharded K1 + peer gather of the tables when every pair of distinct devices has
 * peer access (device k uploads and preprocesses its share of [X | Y], X's part, Y's part or both), otherwise every
 * device uploads X and Y and preprocesses all columns.
 *   Pairs: device k copies the results of its slice straight into the caller's arrays, at its offset from pair_lo.
 *   Edges: as icikt_all_pairs_edges_multi; rows are joined in slice order, which is cross order.
 *   Top-k: every device keeps the lists of the requested sides (rows [c_lo, c_hi) of [X | Y], L = c_hi - c_lo) for
 *   its slice; then device k merges rows [L*k/N, L*(k+1)/N) of all devices' lists, reading them through peer access,
 *   and copies them straight into x_side and / or y_side (a block may hold rows of both).
 *
 *   - Same result as one device: every output (the per-pair arrays, status, rows with their order and fields, cor,
 *     max_taumax, index, n_neighbors, the padding, what icikt_edges_copy returns: j as Y's own index) is bit for bit
 *     that of the matching single-device cross call with the same arguments.
 *   - devices == NULL means ordinals 0..n_devices-1; repeated ordinals are allowed; 1 <= n_devices <= 16.
 *     opts->device is ignored.
 *   - Refused with ICIKT_ERR_BAD_ARG before any device is touched: whatever the single-device cross call refuses
 *     (with the same messages, CSC ones naming the matrix and the column), and n_devices out of range.
 *   - pair_lo / pair_hi: icikt_cross_pairs_multi takes them as icikt_cross_pairs does (the arrays are indexed from
 *     0 = pair_lo); the edges and top-k calls refuse them.
 *   - Peer access: the pairs and edges calls need none.  The top-k call needs it between distinct devices; without
 *     it it runs icikt_cross_topk on devices[0].  With n_devices == 1 each call is its single-device call on
 *     devices[0].
 *   - max_edges: as icikt_all_pairs_edges_multi (the rows held are counted over all devices; once one device crosses
 *     the limit, the others stop at their next window boundary).
 *   - timings (may be NULL): the slowest device's figures, n_launches summed over the devices; for top-k, d2h_ms is
 *     the merge of the device's block with its copy out. */
int icikt_cross_pairs_multi(const icikt_input* x, const icikt_input* y, int64_t n, const double* global_na,
                            int32_t n_global_na, const icikt_opts* opts, const int32_t* devices, int32_t n_devices,
                            double* raw, double* pvalue, double* taumax, double* completeness, int32_t* status,
                            double* max_taumax, icikt_timings* timings);
int icikt_cross_edges_multi(const icikt_input* x, const icikt_input* y, int64_t n, const double* global_na,
                            int32_t n_global_na, const icikt_opts* opts, const int32_t* devices, int32_t n_devices,
                            const icikt_edge_filter* filter, icikt_edges** out, double* max_taumax,
                            icikt_timings* timings);
int icikt_cross_topk_multi(const icikt_input* x, const icikt_input* y, int64_t n, const double* global_na,
                           int32_t n_global_na, const icikt_opts* opts, const int32_t* devices, int32_t n_devices,
                           int32_t k, int32_t by, int32_t scale_max, const icikt_topk_lists* x_side,
                           const icikt_topk_lists* y_side, double* max_taumax, icikt_timings* timings);

/* ---- filtered calls with p-values adjusted over every pair: R's p.adjust(p_all, method), computed on the device window
 * by window without holding P of anything, where p_all is the per-pair p-value array of icikt_all_pairs /
 * icikt_cross_pairs.  Methods are R's bonferroni, holm, hochberg, BH (fdr) and BY; Hommel is not offered (its adjusted
 * values depend on the whole order, not on a prefix).
 *
 *   - Family: every pair of the call's order whose p-value is not NaN, whatever its status: the combn order plus the
 *     diagonal pairs when include_diag is set, or the Cx * Cy cross order.  m, their number, is what p.adjust's n is
 *     after it drops the NAs.  The family does not depend on min_abs_cor or max_pvalue.
 *   - Row predicate: that of icikt_all_pairs_edges / icikt_cross_edges AND (isnan(max_padj) || padj <= max_padj).
 *     Rows, their order, every existing field and max_taumax are bit for bit what those calls return for the same
 *     pairs; padj (icikt_edges_copy_padj) is bit for bit p.adjust(p_all, method) at the row's pair.
 *   - Exactness without every p-value: each multiplier of p.adjust is >= 1 after rounding, so padj >= p, and the
 *     p-values <= max_padj are a prefix of the ascending order whose adjusted values <= max_padj depend only on that
 *     prefix and on m.  Each device keeps one 8-byte key per pair with p <= max_padj (every non-NaN p-value when
 *     max_padj is NaN or >= 1: 8 B per pair) and a count of the non-NaN p-values; after the last window the keys are
 *     gathered on devices[0] (peer copies when every pair of devices has peer access, otherwise through pinned host
 *     memory), sorted and scanned once, and every row finds its value by a binary search of its p-value.  BY's
 *     q = sum(1/(1:m)) is summed on the host in long double, as R's sum does (m steps).  m <= 1 leaves padj = p.
 *   - Refused with ICIKT_ERR_BAD_ARG before any device is touched: whatever the matching edges call refuses, a NULL
 *     adjust, a method out of range, reserved != 0.  The all-pairs calls take the matrix as an icikt_input, dense or
 *     CSC, whose messages name it matrix x.
 *   - max_edges counts the rows held, as in the edges calls (rows are held only when p <= max_padj too); the final
 *     count is taken after the trim with padj.
 *   - timings as in the edges calls; the candidates' pass, the gather, sort, scan and lookup are counted in
 *     epilogue_ms, and total_ms ends with the lookup.  The _multi twins take (devices, n_devices) after opts, as the
 *     edges multi calls, and return bit for bit the single-device result (padj depends only on the p-values and m). */
#define ICIKT_PADJ_BONFERRONI 1
#define ICIKT_PADJ_HOLM 2
#define ICIKT_PADJ_HOCHBERG 3
#define ICIKT_PADJ_BH 4 /* R's "BH" and "fdr" */
#define ICIKT_PADJ_BY 5

typedef struct icikt_padj_filter {
  int32_t method;   /* ICIKT_PADJ_*                                  */
  int32_t reserved; /* 0                                             */
  double max_padj;  /* NaN: no condition on the adjusted p-value     */
} icikt_padj_filter;

/* R's p.adjust(p[0..m), method) on the device: NaN entries are dropped from the family and stay as they are (their
 * bits), *n_tests (may be NULL) receives the number of non-NaN entries, and fewer than two of them leave p unchanged.
 * -0.0 counts as +0.0.  p and out may be NULL when m == 0.  Refused with ICIKT_ERR_BAD_ARG: m < 0, NULL p / out with
 * m > 0, a method out of range.  Device memory: about 56 B per entry. */
int icikt_p_adjust(const double* p, int64_t m, int32_t method, int32_t device, double* out, int64_t* n_tests);

int icikt_all_pairs_edges_padj(const icikt_input* x, int64_t n, const double* global_na, int32_t n_global_na,
                               const icikt_opts* opts, const icikt_edge_filter* filter, const icikt_padj_filter* adjust,
                               icikt_edges** out, double* max_taumax, icikt_timings* timings);
int icikt_all_pairs_edges_padj_multi(const icikt_input* x, int64_t n, const double* global_na, int32_t n_global_na,
                                     const icikt_opts* opts, const int32_t* devices, int32_t n_devices,
                                     const icikt_edge_filter* filter, const icikt_padj_filter* adjust, icikt_edges** out,
                                     double* max_taumax, icikt_timings* timings);
int icikt_cross_edges_padj(const icikt_input* x, const icikt_input* y, int64_t n, const double* global_na,
                           int32_t n_global_na, const icikt_opts* opts, const icikt_edge_filter* filter,
                           const icikt_padj_filter* adjust, icikt_edges** out, double* max_taumax,
                           icikt_timings* timings);
int icikt_cross_edges_padj_multi(const icikt_input* x, const icikt_input* y, int64_t n, const double* global_na,
                                 int32_t n_global_na, const icikt_opts* opts, const int32_t* devices, int32_t n_devices,
                                 const icikt_edge_filter* filter, const icikt_padj_filter* adjust, icikt_edges** out,
                                 double* max_taumax, icikt_timings* timings);
/* the adjusted p-values of a _padj result into padj[icikt_edges_count(e)]; ICIKT_ERR_BAD_ARG for a result without */
int icikt_edges_copy_padj(const icikt_edges* e, double* padj);
/* m of a _padj result; -1 for NULL or a result without adjustment */
int64_t icikt_edges_n_tests(const icikt_edges* e);

/* ---- edge counts: how many pairs pass each of several edge filters, and each column's degree under each, in ONE walk
 * of the pair order and without returning a single pair -- what a threshold would return before the filtered call is
 * run with it (edges against threshold, degree distributions, hub and isolated columns).  The pair kernel runs once
 * whatever the number of filters.
 *
 *   - Input: that of the filtered calls, all pairs of one matrix (an icikt_input, dense or CSC, whose messages name it
 *     matrix x; the diagonal pairs follow when include_diag is set) or the cross order of X against Y.
 *   - Filters: filters[0 .. n_filters), 1 <= n_filters <= ICIKT_COUNT_FILTERS_MAX, each an icikt_edge_filter with
 *     scale_max = 0, reserved = 0 and max_edges = 0.  A pair passes filter f under exactly the predicate of
 *     icikt_all_pairs_edges without scale_max: status == 0 && (isnan(min_abs_cor) || fabs(raw) >= min_abs_cor) &&
 *     (isnan(max_pvalue) || pvalue <= max_pvalue).  Scaled thresholds are refused: whether a pair passes raw / M >= t
 *     depends on M = max(taumax), known only after the last window, and a count has no rows to trim once it is.  The
 *     call returns M in max_taumax, so a scaled threshold t is counted as the raw threshold t * M.  That is the
 *     meaning of scaling here; it can differ from scale_max = 1 (fabs(raw / M) >= t) in the last ulp at the boundary.
 *   - Outputs, caller-allocated: n_pass[T] (required) the pairs that pass each filter, icikt_edges_count of the
 *     filtered call with that one filter; degree[C * T] (may be NULL), entry c * T + f, the passing pairs of filter f
 *     that have column c as either endpoint, a diagonal pair (c, c) counting once; for a cross call x_degree[Cx * T]
 *     and y_degree[Cy * T] (each may be NULL) the same over X's and Y's columns; status_counts[ICIKT_NSTATUS] (may be
 *     NULL) the pairs per status class, as icikt_matrices returns them; max_taumax (may be NULL) M or NaN.
 *   - Every output is an integer count independent of the order of the work, so the _multi twins ((devices, n_devices)
 *     after opts, as the edges multi calls; per-device counts summed on the host) return bit for bit the one-device
 *     result.
 *   - Device memory does not depend on the number of pairs: the per-column tables, one window of pairs
 *     (ICIKT_EDGE_WINDOW) and 8 B x (C x T + T + 16) of counters, which come back once, after the last window.
 *   - Refused with ICIKT_ERR_BAD_ARG before any device is touched: n_filters out of range, a NULL filters or n_pass, a
 *     filter with scale_max, max_edges or reserved != 0, and whatever the filtered call refuses of its options
 *     (ICIKT_PERSPECTIVE_COMPLETE, ICIKT_KERNEL_NAIVE, want_counts, pair_lo / pair_hi != 0; for cross calls
 *     include_diag), n_devices out of 1..16.
 *   - timings (may be NULL) as in the edges calls: epilogue_ms includes the counting pass, d2h_ms is the copy of the
 *     counters. */
#define ICIKT_COUNT_FILTERS_MAX 64

int icikt_all_pairs_count_edges(const icikt_input* x, int64_t n, const double* global_na, int32_t n_global_na,
                                const icikt_opts* opts, const icikt_edge_filter* filters, int32_t n_filters,
                                int64_t* n_pass, int64_t* degree, int64_t* status_counts, double* max_taumax,
                                icikt_timings* timings);
int icikt_all_pairs_count_edges_multi(const icikt_input* x, int64_t n, const double* global_na, int32_t n_global_na,
                                      const icikt_opts* opts, const int32_t* devices, int32_t n_devices,
                                      const icikt_edge_filter* filters, int32_t n_filters, int64_t* n_pass,
                                      int64_t* degree, int64_t* status_counts, double* max_taumax,
                                      icikt_timings* timings);
int icikt_cross_count_edges(const icikt_input* x, const icikt_input* y, int64_t n, const double* global_na,
                            int32_t n_global_na, const icikt_opts* opts, const icikt_edge_filter* filters,
                            int32_t n_filters, int64_t* n_pass, int64_t* x_degree, int64_t* y_degree,
                            int64_t* status_counts, double* max_taumax, icikt_timings* timings);
int icikt_cross_count_edges_multi(const icikt_input* x, const icikt_input* y, int64_t n, const double* global_na,
                                  int32_t n_global_na, const icikt_opts* opts, const int32_t* devices,
                                  int32_t n_devices, const icikt_edge_filter* filters, int32_t n_filters,
                                  int64_t* n_pass, int64_t* x_degree, int64_t* y_degree, int64_t* status_counts,
                                  double* max_taumax, icikt_timings* timings);

/* ---- plan API: keeps the matrix, the per-column tables and the results resident in
 * HBM so that repeated runs (benchmarks, several perspectives on one matrix) do not
 * pay the copies.  A plan is bound to one device and is not thread-safe.            */
typedef struct icikt_plan icikt_plan;

/* pi/pj NULL => all pairs (honours opts->include_diag, pair_lo/pair_hi).            */
int icikt_plan_create(icikt_plan** plan, int64_t n, int64_t C, const int32_t* pi,
                      const int32_t* pj, int64_t P, const icikt_opts* opts);
int64_t icikt_plan_num_pairs(const icikt_plan* plan);
/* copy the host matrix into the plan's device buffer (pinned staging inside)        */
int icikt_plan_upload(icikt_plan* plan, const double* data, int64_t ld);
/* or hand over a device pointer (column-major, ld), e.g. a torch tensor's data_ptr  */
int icikt_plan_set_device_matrix(icikt_plan* plan, const double* d_data, int64_t ld);
/* K1: missing marking, sort, dense ranks, tie sums, per-column tables               */
int icikt_plan_columns(icikt_plan* plan, const double* global_na, int32_t n_global_na);
/* Sharded K1 (one process or worker per GPU, SURVEY.md 8e): the per-column work of columns
 * [col_lo, col_hi) only.  A rank uploads and preprocesses its slice of the columns, the ranks
 * exchange the table slices icikt_plan_tables describes (column c of table k lives at
 * ptr + c * bytes_per_column, on the plan's device; any transport: NCCL all-gather, peer
 * copies), then icikt_plan_columns_finish derives the launch tier from the statistics of all
 * columns and releases icikt_plan_pairs.  `data`/`ld` address the whole matrix.            */
typedef struct icikt_table {
  void* ptr;                /* device pointer to column 0 of the table */
  int64_t bytes_per_column;
} icikt_table;
#define ICIKT_MAX_TABLES 16
int icikt_plan_upload_columns(icikt_plan* plan, const double* data, int64_t ld, int64_t col_lo,
                              int64_t col_hi);
int icikt_plan_columns_range(icikt_plan* plan, const double* global_na, int32_t n_global_na,
                             int64_t col_lo, int64_t col_hi);
/* fills out[0..min(cap, n)) and returns n, the number of tables to exchange (<= ICIKT_MAX_TABLES) */
int icikt_plan_tables(icikt_plan* plan, icikt_table* out, int32_t cap);
int icikt_plan_columns_finish(icikt_plan* plan);
/* K2+K3 over the plan's pairs; results stay on the device                           */
int icikt_plan_pairs(icikt_plan* plan);
/* block until the plan's stream is idle                                             */
int icikt_plan_sync(icikt_plan* plan);
/* copy results to host arrays (any may be NULL)                                     */
int icikt_plan_download(icikt_plan* plan, double* raw, double* pvalue, double* taumax,
                        double* completeness, int32_t* status, int64_t* counts,
                        double* max_taumax);
/* scale_and_reshape (R/kendalltau.R:357-421) on the device: the results of the plan's pairs as
 * symmetric C x C column-major matrices (each may be NULL): cor = raw / max(taumax) if scale_max
 * else raw (:368-372); entries without a computed pair are 0 (:389-396); if diag_good the diagonal
 * is n_good/max(n_good) in cor and raw, 0 in pvalue, 1 in taumax, n_good/n in completeness
 * (:374-386) with n_good[C] from the caller or, if NULL, n minus the column's missing count.
 * Degenerate pairs (status != 0) hold the NaN with R's NA_real_ bit pattern 0x7FF00000000007A2 in all
 * five matrices; status_counts[ICIKT_NSTATUS] (may be NULL) receives the number of pairs per status
 * class so that the host can raise each warning once.                                     */
int icikt_plan_download_matrices(icikt_plan* plan, int32_t scale_max, int32_t diag_good,
                                 const int32_t* n_good, double* cor, double* raw, double* pvalue,
                                 double* taumax, double* completeness, int64_t* status_counts,
                                 double* max_taumax);
/* per-column by-products: n_na[C] (missing count per column, gives n_good and
 * frac_complete of R/kendalltau.R:165-167); may be NULL                             */
int icikt_plan_column_info(icikt_plan* plan, int32_t* n_na);
/* the CUDA stream the plan launches on, as a cudaStream_t cast to void*             */
void* icikt_plan_stream(icikt_plan* plan);
/* timings of the last upload/columns/pairs/download calls                           */
int icikt_plan_timings(icikt_plan* plan, icikt_timings* t);
void icikt_plan_destroy(icikt_plan* plan);

/* Standard normal CDF exactly as the epilogue kernel evaluates it (R nmath pnorm
 * semantics incl. the exact-zero tails), computed ON THE DEVICE for n values.
 * Test hook for the p-value path; lower_tail as in pnorm().                         */
int icikt_pnorm_device(const double* z, int64_t n, int32_t lower_tail, double* out,
                       int32_t device);

/* Host-only helper: the (i, j) columns of pair `index` in the pair order of icikt_all_pairs
 * (utils::combn(C, 2) order, then the diagonal if include_diag).  Used by callers that shard
 * the pair order with pair_lo/pair_hi or scatter results into C x C matrices.             */
int icikt_pair_from_index(int64_t C, int32_t include_diag, int64_t index, int32_t* i, int32_t* j);

/* The one-shot calls keep their device workspace (tables, result buffers, stream) cached
 * between calls with the same shape so that repeated calls do not pay cudaMalloc; this
 * frees it (the R shim calls it from .onUnload).                                      */
void icikt_release_workspace(void);

/* How the one-shot calls (icikt_all_pairs, icikt_matrices) pipeline a large all-pairs job (input of
 * ICIKT_PIPELINE_MIN_BYTES = 32 MB or more, 128 columns or more; ICIKT_NO_PIPELINE=1 switches it off).
 * The reference hands each furrr worker the whole matrix and a slice of the pair list (R/kendalltau.R:
 * 236-253); here the columns are uploaded in chunks [0,f), [f,2f), [2f,4f) ... and the launch that follows a
 * chunk computes every pair whose later column lies in it, so the upload of the next chunk hides behind
 * it; the last chunk is cut into n_blocks row blocks whose results are contiguous in the pair order and
 * are copied out while the next block runs.  This host-only function reports that table for C columns:
 * units[4k..] = (slot, first column, other column of its first pair, pairs), launches[6l..] = (col_lo,
 * col_hi, unit_lo, unit_hi, slot_lo, slot_hi); cta_slots = resident CTAs of the pair kernel (2 x SMs).
 * Returns the number of units (or a negative error); at most cap_units / cap_launches entries are
 * written (either array may be NULL).  Needs no device.                                         */
int64_t icikt_stage_table(int64_t C, int32_t include_diag, int32_t cta_slots, int32_t n_blocks,
                          int64_t cap_units, int64_t* units, int64_t cap_launches, int64_t* launches,
                          int64_t* n_launches);

/* The pair kernel's launch shape for vectors of n rows (host only, no device needed; what the plan selects
 * in icikt_plan_columns): tier 0 / 1 / 2 = no large tie groups / large groups sorted in place / pass B.
 * out[0] warps per CTA, out[1] 8-key runs per thread, out[2] bytes of the per-CTA region (sequence buffers +
 * counter area), out[3] variant (0 two sequence buffers in shared memory, 1 in place, 2 global scratch),
 * out[4] padded length (keys), out[5] in place: rows per staging part of the gather, out[6] 1 if pass A runs
 * radix-16 levels below its top bits (chosen by n alone).  n_sm = SMs of the device (148), complete_obs != 0
 * for the complete-observations mode.                                                                     */
int icikt_launch_shape(int64_t n, int32_t tier, int32_t n_sm, int32_t complete_obs, int32_t* out);

/* Measures the shared-memory bandwidth of `device` with a conflict-free read+write sweep
 * (the traffic pattern the roofline model of the pair kernel assumes: one 32-bit load and
 * one 32-bit store per element per level).  Returns GB/s through the pointers (either may
 * be NULL): 32-bit accesses and 128-bit accesses.  Benchmark utility, not on the hot path. */
int icikt_measure_smem_bandwidth(int32_t device, double* gbps_32bit, double* gbps_128bit);

/* Measures the sustained instruction-issue rate of `device`, in G warp-instructions per second over
 * the whole GPU, for the two pipes the pair kernel lives on: LOP3 only (integer ALU pipe), IMAD only
 * (FMA pipe), and the two interleaved (what a kernel that balances them can reach).  The pair
 * kernel's executed warp instructions divided by its run time, over the interleaved figure, is the
 * INT/issue roofline fraction bench.py prints.  Any pointer may be NULL.                        */
int icikt_measure_issue_rate(int32_t device, double* alu_only, double* fma_only, double* interleaved);

#ifdef __cplusplus
}
#endif
#endif /* ICIKT_B200_H */
