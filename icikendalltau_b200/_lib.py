"""ctypes binding of libicikt_b200.so (the C ABI in include/icikt_b200.h).

The library is the product's only compute path.  If it is missing, or no CUDA device is
usable, every call raises -- there is no CPU fallback.
"""
from __future__ import annotations

import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# ICIKT_LIB_PATH: another build of the same library (A/B runs of tuning variants); default: the in-tree build
LIB_PATH = os.environ.get("ICIKT_LIB_PATH") or os.path.join(_HERE, "libicikt_b200.so")

OK = 0
ERR_NO_DEVICE, ERR_BAD_ARG, ERR_TOO_LONG, ERR_CUDA, ERR_ALLOC, ERR_LIMIT = -1, -2, -3, -4, -5, -6
NCOUNTS = 7
TOPK_BY = {"abs": 0, "signed": 1}
TOPK_MAX = 1024
COUNT_FILTERS_MAX = 64
KERNEL_TILED, KERNEL_NAIVE = 0, 1
PERSPECTIVE = {"global": 0, "local": 1, "complete": 2}
ALTERNATIVE = {"two.sided": 0, "less": 1, "greater": 2}
# R's p.adjust methods offered (ICIKT_PADJ_*); "fdr" is R's alias of "BH", "hommel" is not offered
PADJ = {"bonferroni": 1, "holm": 2, "hochberg": 3, "BH": 4, "fdr": 4, "BY": 5}

# every symbol include/icikt_b200.h declares (checked by tests/test_abi_cpu.py)
EXPORTS = [
    "icikt_default_opts", "icikt_abi_version", "icikt_device_count", "icikt_max_n",
    "icikt_last_error", "icikt_all_pairs", "icikt_pair_list", "icikt_plan_create",
    "icikt_plan_num_pairs", "icikt_plan_upload", "icikt_plan_set_device_matrix",
    "icikt_plan_columns", "icikt_plan_pairs", "icikt_plan_sync", "icikt_plan_download",
    "icikt_plan_column_info", "icikt_plan_stream", "icikt_plan_timings", "icikt_plan_destroy",
    "icikt_pnorm_device", "icikt_release_workspace", "icikt_measure_smem_bandwidth",
    "icikt_pair_from_index", "icikt_all_pairs_multi", "icikt_matrices", "icikt_plan_download_matrices",
    "icikt_pairwise_completeness", "icikt_plan_upload_columns", "icikt_plan_columns_range",
    "icikt_plan_tables", "icikt_plan_columns_finish", "icikt_measure_issue_rate",
    "icikt_matrices_multi", "icikt_stage_table", "icikt_launch_shape",
    "icikt_all_pairs_csc", "icikt_all_pairs_multi_csc", "icikt_pair_list_csc", "icikt_matrices_csc",
    "icikt_matrices_multi_csc", "icikt_pairwise_completeness_csc",
    "icikt_all_pairs_edges", "icikt_all_pairs_edges_csc", "icikt_edges_count", "icikt_edges_copy",
    "icikt_edges_free", "icikt_all_pairs_topk", "icikt_all_pairs_topk_csc",
    "icikt_all_pairs_edges_multi", "icikt_all_pairs_edges_multi_csc", "icikt_all_pairs_topk_multi",
    "icikt_all_pairs_topk_multi_csc", "icikt_cross_pairs", "icikt_cross_edges", "icikt_cross_topk",
    "icikt_cross_pairs_multi", "icikt_cross_edges_multi", "icikt_cross_topk_multi",
    "icikt_p_adjust", "icikt_all_pairs_edges_padj", "icikt_all_pairs_edges_padj_multi", "icikt_cross_edges_padj",
    "icikt_cross_edges_padj_multi", "icikt_edges_copy_padj", "icikt_edges_n_tests",
    "icikt_all_pairs_count_edges", "icikt_all_pairs_count_edges_multi", "icikt_cross_count_edges",
    "icikt_cross_count_edges_multi",
]
NSTATUS = 10


class IciktError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libicikt_b200 error {code}: {msg}")
        self.code = code


class Opts(ctypes.Structure):
    _fields_ = [("perspective", ctypes.c_int32), ("alternative", ctypes.c_int32),
                ("continuity", ctypes.c_int32), ("include_diag", ctypes.c_int32),
                ("na_inf", ctypes.c_int32), ("device", ctypes.c_int32),
                ("kernel", ctypes.c_int32), ("want_counts", ctypes.c_int32),
                ("pair_lo", ctypes.c_int64), ("pair_hi", ctypes.c_int64)]


class Timings(ctypes.Structure):
    _fields_ = [("h2d_ms", ctypes.c_float), ("columns_ms", ctypes.c_float),
                ("pairs_ms", ctypes.c_float), ("epilogue_ms", ctypes.c_float), ("d2h_ms", ctypes.c_float),
                ("total_ms", ctypes.c_float), ("n_launches", ctypes.c_int32),
                ("reserved", ctypes.c_int32)]

    def as_dict(self):
        return dict(h2d_ms=self.h2d_ms, columns_ms=self.columns_ms, pairs_ms=self.pairs_ms,
                    epilogue_ms=self.epilogue_ms, d2h_ms=self.d2h_ms, total_ms=self.total_ms,
                    n_launches=self.n_launches)


class EdgeFilter(ctypes.Structure):
    _fields_ = [("min_abs_cor", ctypes.c_double), ("max_pvalue", ctypes.c_double),
                ("scale_max", ctypes.c_int32), ("reserved", ctypes.c_int32), ("max_edges", ctypes.c_int64)]


class PadjFilter(ctypes.Structure):
    _fields_ = [("method", ctypes.c_int32), ("reserved", ctypes.c_int32), ("max_padj", ctypes.c_double)]


class Input(ctypes.Structure):
    """icikt_input: one matrix of a cross call, dense (data, ld) or CSC (colptr, rowidx, values)."""
    _fields_ = [("C", ctypes.c_int64), ("data", ctypes.c_void_p), ("ld", ctypes.c_int64),
                ("colptr", ctypes.c_void_p), ("rowidx", ctypes.c_void_p), ("values", ctypes.c_void_p)]


class TopkLists(ctypes.Structure):
    """icikt_topk_lists: the caller arrays of one side of icikt_cross_topk."""
    _fields_ = [("index", ctypes.c_void_p), ("n_neighbors", ctypes.c_void_p), ("cor", ctypes.c_void_p),
                ("raw", ctypes.c_void_p), ("pvalue", ctypes.c_void_p), ("taumax", ctypes.c_void_p),
                ("completeness", ctypes.c_void_p)]


class Table(ctypes.Structure):
    _fields_ = [("ptr", ctypes.c_void_p), ("bytes_per_column", ctypes.c_int64)]


MAX_TABLES = 16

_lib = None
# array arguments travel as plain addresses (void*): building typed ctypes pointers from NumPy
# arrays costs microseconds each, which shows in the one-shot call on small matrices
_dp = _ip = _lp = ctypes.c_void_p


def load():
    """Load the shared library; raises if it has not been built (python -m icikendalltau_b200.build)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise IciktError(ERR_NO_DEVICE, f"{LIB_PATH} is missing: build it with "
                         "`python -m icikendalltau_b200.build` (nvcc, sm_100a); there is no CPU fallback")
    L = ctypes.CDLL(LIB_PATH)
    vp = ctypes.c_void_p
    L.icikt_default_opts.argtypes = [ctypes.POINTER(Opts)]
    L.icikt_default_opts.restype = None
    L.icikt_abi_version.restype = ctypes.c_int
    L.icikt_device_count.restype = ctypes.c_int
    L.icikt_max_n.restype = ctypes.c_int64
    L.icikt_last_error.restype = ctypes.c_char_p
    common_out = [_dp, _dp, _dp, _dp, _ip, _lp, _dp, ctypes.POINTER(Timings)]
    L.icikt_all_pairs.argtypes = [_dp, ctypes.c_int64, ctypes.c_int64, ctypes.c_int64, _dp,
                                  ctypes.c_int32, ctypes.POINTER(Opts)] + common_out
    L.icikt_all_pairs.restype = ctypes.c_int
    L.icikt_all_pairs_multi.argtypes = [_dp, ctypes.c_int64, ctypes.c_int64, ctypes.c_int64, _dp,
                                        ctypes.c_int32, ctypes.POINTER(Opts), _ip, ctypes.c_int32] + common_out
    L.icikt_all_pairs_multi.restype = ctypes.c_int
    L.icikt_pair_list.argtypes = [_dp, ctypes.c_int64, ctypes.c_int64, ctypes.c_int64, _dp,
                                  ctypes.c_int32, _ip, _ip, ctypes.c_int64,
                                  ctypes.POINTER(Opts)] + common_out
    L.icikt_pair_list.restype = ctypes.c_int
    L.icikt_plan_create.argtypes = [ctypes.POINTER(vp), ctypes.c_int64, ctypes.c_int64, _ip, _ip,
                                    ctypes.c_int64, ctypes.POINTER(Opts)]
    L.icikt_plan_create.restype = ctypes.c_int
    L.icikt_plan_num_pairs.argtypes = [vp]
    L.icikt_plan_num_pairs.restype = ctypes.c_int64
    L.icikt_plan_upload.argtypes = [vp, _dp, ctypes.c_int64]
    L.icikt_plan_upload.restype = ctypes.c_int
    L.icikt_plan_set_device_matrix.argtypes = [vp, vp, ctypes.c_int64]
    L.icikt_plan_set_device_matrix.restype = ctypes.c_int
    L.icikt_plan_columns.argtypes = [vp, _dp, ctypes.c_int32]
    L.icikt_plan_columns.restype = ctypes.c_int
    L.icikt_plan_upload_columns.argtypes = [vp, _dp, ctypes.c_int64, ctypes.c_int64, ctypes.c_int64]
    L.icikt_plan_upload_columns.restype = ctypes.c_int
    L.icikt_plan_columns_range.argtypes = [vp, _dp, ctypes.c_int32, ctypes.c_int64, ctypes.c_int64]
    L.icikt_plan_columns_range.restype = ctypes.c_int
    L.icikt_plan_tables.argtypes = [vp, ctypes.POINTER(Table), ctypes.c_int32]
    L.icikt_plan_tables.restype = ctypes.c_int
    L.icikt_plan_columns_finish.argtypes = [vp]
    L.icikt_plan_columns_finish.restype = ctypes.c_int
    L.icikt_plan_pairs.argtypes = [vp]
    L.icikt_plan_pairs.restype = ctypes.c_int
    L.icikt_plan_sync.argtypes = [vp]
    L.icikt_plan_sync.restype = ctypes.c_int
    L.icikt_plan_download.argtypes = [vp, _dp, _dp, _dp, _dp, _ip, _lp, _dp]
    L.icikt_plan_download.restype = ctypes.c_int
    L.icikt_plan_download_matrices.argtypes = [vp, ctypes.c_int32, ctypes.c_int32, _ip, _dp, _dp, _dp, _dp, _dp,
                                               _lp, _dp]
    L.icikt_plan_download_matrices.restype = ctypes.c_int
    L.icikt_matrices.argtypes = [_dp, ctypes.c_int64, ctypes.c_int64, ctypes.c_int64, _dp, ctypes.c_int32,
                                 _ip, _ip, ctypes.c_int64, ctypes.POINTER(Opts), ctypes.c_int32, ctypes.c_int32,
                                 _ip, _dp, _dp, _dp, _dp, _dp, _lp, _dp, ctypes.POINTER(Timings)]
    L.icikt_matrices.restype = ctypes.c_int
    L.icikt_matrices_multi.argtypes = [_dp, ctypes.c_int64, ctypes.c_int64, ctypes.c_int64, _dp, ctypes.c_int32,
                                       ctypes.POINTER(Opts), _ip, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32,
                                       _ip, _dp, _dp, _dp, _dp, _dp, _lp, _dp, ctypes.POINTER(Timings)]
    L.icikt_matrices_multi.restype = ctypes.c_int
    L.icikt_pairwise_completeness.argtypes = [_dp, ctypes.c_int64, ctypes.c_int64, ctypes.c_int64, _dp,
                                              ctypes.c_int32, ctypes.c_int32, _ip, _ip, ctypes.c_int64, _ip,
                                              _dp, _dp]
    L.icikt_pairwise_completeness.restype = ctypes.c_int
    # the *_csc twins: (data, n, C, ld) -> (colptr, rowidx, values, n, C)
    csc = [_lp, _ip, _dp, ctypes.c_int64, ctypes.c_int64]
    for name in ("icikt_all_pairs", "icikt_all_pairs_multi", "icikt_pair_list", "icikt_matrices",
                 "icikt_matrices_multi", "icikt_pairwise_completeness"):
        f = getattr(L, name + "_csc")
        f.argtypes = csc + getattr(L, name).argtypes[4:]
        f.restype = ctypes.c_int
    L.icikt_all_pairs_edges.argtypes = [_dp, ctypes.c_int64, ctypes.c_int64, ctypes.c_int64, _dp, ctypes.c_int32,
                                        ctypes.POINTER(Opts), ctypes.POINTER(EdgeFilter), ctypes.POINTER(vp), _dp,
                                        ctypes.POINTER(Timings)]
    L.icikt_all_pairs_edges.restype = ctypes.c_int
    L.icikt_all_pairs_edges_csc.argtypes = csc + L.icikt_all_pairs_edges.argtypes[4:]
    L.icikt_all_pairs_edges_csc.restype = ctypes.c_int
    L.icikt_edges_count.argtypes = [vp]
    L.icikt_edges_count.restype = ctypes.c_int64
    L.icikt_edges_copy.argtypes = [vp, _ip, _ip, _dp, _dp, _dp, _dp, _dp]
    L.icikt_edges_copy.restype = ctypes.c_int
    L.icikt_edges_free.argtypes = [vp]
    L.icikt_edges_free.restype = None
    L.icikt_all_pairs_topk.argtypes = [_dp, ctypes.c_int64, ctypes.c_int64, ctypes.c_int64, _dp, ctypes.c_int32,
                                       ctypes.POINTER(Opts), ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, _ip, _ip,
                                       _dp, _dp, _dp, _dp, _dp, _dp, ctypes.POINTER(Timings)]
    L.icikt_all_pairs_topk.restype = ctypes.c_int
    L.icikt_all_pairs_topk_csc.argtypes = csc + L.icikt_all_pairs_topk.argtypes[4:]
    L.icikt_all_pairs_topk_csc.restype = ctypes.c_int
    # the multi-device twins of the filtered calls: (devices, n_devices) after opts
    for name in ("icikt_all_pairs_edges", "icikt_all_pairs_topk"):
        a = getattr(L, name).argtypes
        for sfx, lead in (("_multi", a[:7]), ("_multi_csc", csc + a[4:7])):
            f = getattr(L, name + sfx)
            f.argtypes = lead + [_ip, ctypes.c_int32] + a[7:]
            f.restype = ctypes.c_int
    cross = [ctypes.POINTER(Input), ctypes.POINTER(Input), ctypes.c_int64, _dp, ctypes.c_int32, ctypes.POINTER(Opts)]
    L.icikt_cross_pairs.argtypes = cross + [_dp, _dp, _dp, _dp, _ip, _dp, ctypes.POINTER(Timings)]
    L.icikt_cross_pairs.restype = ctypes.c_int
    L.icikt_cross_edges.argtypes = cross + L.icikt_all_pairs_edges.argtypes[7:]
    L.icikt_cross_edges.restype = ctypes.c_int
    L.icikt_cross_topk.argtypes = cross + [ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, ctypes.POINTER(TopkLists),
                                           ctypes.POINTER(TopkLists), _dp, ctypes.POINTER(Timings)]
    L.icikt_cross_topk.restype = ctypes.c_int
    for name in ("icikt_cross_pairs", "icikt_cross_edges", "icikt_cross_topk"):  # (devices, n_devices) after opts
        a = getattr(L, name).argtypes
        f = getattr(L, name + "_multi")
        f.argtypes = a[:6] + [_ip, ctypes.c_int32] + a[6:]
        f.restype = ctypes.c_int
    # the _padj twins of the edges calls: the matrix as an icikt_input, the icikt_padj_filter after the edge filter
    ef = [ctypes.POINTER(EdgeFilter), ctypes.POINTER(PadjFilter), ctypes.POINTER(vp), _dp, ctypes.POINTER(Timings)]
    one = [ctypes.POINTER(Input), ctypes.c_int64, _dp, ctypes.c_int32, ctypes.POINTER(Opts)]
    for name, lead in (("icikt_all_pairs_edges_padj", one), ("icikt_cross_edges_padj", cross)):
        getattr(L, name).argtypes = lead + ef
        getattr(L, name + "_multi").argtypes = lead + [_ip, ctypes.c_int32] + ef
        getattr(L, name).restype = getattr(L, name + "_multi").restype = ctypes.c_int
    # the edge-count calls: (filters, n_filters, n_pass, degree or x_degree + y_degree, status_counts, max_taumax,
    # timings) after opts, or after (devices, n_devices) for the _multi twins
    cnt = [ctypes.POINTER(EdgeFilter), ctypes.c_int32, _lp]
    tail = [_lp, _dp, ctypes.POINTER(Timings)]
    for name, lead, deg in (("icikt_all_pairs_count_edges", one, [_lp]), ("icikt_cross_count_edges", cross, [_lp, _lp])):
        getattr(L, name).argtypes = lead + cnt + deg + tail
        getattr(L, name + "_multi").argtypes = lead + [_ip, ctypes.c_int32] + cnt + deg + tail
        getattr(L, name).restype = getattr(L, name + "_multi").restype = ctypes.c_int
    L.icikt_p_adjust.argtypes = [_dp, ctypes.c_int64, ctypes.c_int32, ctypes.c_int32, _dp, ctypes.POINTER(ctypes.c_int64)]
    L.icikt_p_adjust.restype = ctypes.c_int
    L.icikt_edges_copy_padj.argtypes = [vp, _dp]
    L.icikt_edges_copy_padj.restype = ctypes.c_int
    L.icikt_edges_n_tests.argtypes = [vp]
    L.icikt_edges_n_tests.restype = ctypes.c_int64
    L.icikt_plan_column_info.argtypes = [vp, _ip]
    L.icikt_plan_column_info.restype = ctypes.c_int
    L.icikt_plan_stream.argtypes = [vp]
    L.icikt_plan_stream.restype = vp
    L.icikt_plan_timings.argtypes = [vp, ctypes.POINTER(Timings)]
    L.icikt_plan_timings.restype = ctypes.c_int
    L.icikt_plan_destroy.argtypes = [vp]
    L.icikt_plan_destroy.restype = None
    L.icikt_pnorm_device.argtypes = [_dp, ctypes.c_int64, ctypes.c_int32, _dp, ctypes.c_int32]
    L.icikt_pnorm_device.restype = ctypes.c_int
    L.icikt_pair_from_index.argtypes = [ctypes.c_int64, ctypes.c_int32, ctypes.c_int64, _ip, _ip]
    L.icikt_pair_from_index.restype = ctypes.c_int
    L.icikt_release_workspace.argtypes = []
    L.icikt_release_workspace.restype = None
    L.icikt_measure_smem_bandwidth.argtypes = [ctypes.c_int32, _dp, _dp]
    L.icikt_measure_smem_bandwidth.restype = ctypes.c_int
    L.icikt_measure_issue_rate.argtypes = [ctypes.c_int32, _dp, _dp, _dp]
    L.icikt_measure_issue_rate.restype = ctypes.c_int
    L.icikt_stage_table.argtypes = [ctypes.c_int64, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, ctypes.c_int64,
                                    _lp, ctypes.c_int64, _lp, _lp]
    L.icikt_stage_table.restype = ctypes.c_int64
    L.icikt_launch_shape.argtypes = [ctypes.c_int64, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, _ip]
    L.icikt_launch_shape.restype = ctypes.c_int
    _lib = L
    return L


def check(rc):
    if rc != OK:
        raise IciktError(rc, load().icikt_last_error().decode(errors="replace"))


def make_opts(perspective="global", alternative="two.sided", continuity=False, include_diag=False,
              na_inf=False, device=0, kernel=KERNEL_TILED, want_counts=False, pair_lo=0, pair_hi=0):
    # same values as icikt_default_opts() for everything not given (all zero)
    return Opts(PERSPECTIVE.get(perspective, 0),   # any other string behaves as global
                ALTERNATIVE.get(alternative, 3),   # unknown alternative: p-value stays 0
                int(bool(continuity)), int(bool(include_diag)), int(bool(na_inf)), int(device), int(kernel),
                int(bool(want_counts)), int(pair_lo), int(pair_hi))


def _global_na_array(global_na):
    if len(global_na) == 0:
        return None, None, 0
    g = np.ascontiguousarray(np.asarray(list(global_na), dtype=np.float64))
    return g, _ptr(g), int(g.size)


def _ptr(a, t=None):
    """address of a NumPy array's buffer (None -> NULL); `t` names the element type for the reader"""
    return a.__array_interface__["data"][0] if a is not None else None


def is_sparse(x):
    """True for a scipy.sparse matrix or array (scipy is imported only for objects that may be one)."""
    if not hasattr(x, "tocsc"):
        return False
    import scipy.sparse as sp
    return sp.issparse(x)


def canonical_csc(x):
    """x as a scipy.sparse CSC matrix or array in canonical format (rows sorted and unique within each
    column).  Duplicate entries are summed, as toarray() does, on a copy: the caller's object stays as it is."""
    if getattr(x, "format", None) == "csc" and len(x.shape) == 2:
        # before scipy looks at the arrays: its versions differ in whether, where and with which message they
        # refuse a column pointer array that disagrees with them
        nnz = int(x.indptr[-1]) if x.indptr.size else 0
        if x.indptr.size != x.shape[1] + 1 or x.indices.size < nnz or x.data.size < nnz:
            raise ValueError(f"malformed CSC matrix: {x.indptr.size} column pointers for {x.shape[1]} columns, "
                             f"colptr[C] = {nnz}, {x.indices.size} row indices, {x.data.size} values")
    a = x.tocsc()
    if len(a.shape) != 2:
        raise ValueError("data must be a 2-D array (features x samples)")
    if not a.has_canonical_format:
        a = a.copy()
        a.sum_duplicates()
    return a


class CSC:
    """A sparse matrix as the *_csc entry points take it: colptr int64 [C + 1], rowidx int32 and values
    float64 [nnz] of its canonical CSC form.  Entries not stored are 0.0."""

    def __init__(self, x):
        a = canonical_csc(x)
        self.shape = (int(a.shape[0]), int(a.shape[1]))
        self.colptr = np.ascontiguousarray(a.indptr, dtype=np.int64)
        self.rowidx = np.ascontiguousarray(a.indices, dtype=np.int32)
        self.values = np.ascontiguousarray(a.data, dtype=np.float64)
        nnz = int(self.colptr[-1]) if self.colptr.size else 0
        if self.colptr.size != self.shape[1] + 1 or self.rowidx.size != nnz or self.values.size != nnz:
            raise ValueError(f"malformed CSC matrix: {self.colptr.size} column pointers for {self.shape[1]} columns, "
                             f"colptr[C] = {nnz}, {self.rowidx.size} row indices, {self.values.size} values")

    def args(self):
        """the leading (colptr, rowidx, values, n, C) arguments of a *_csc entry point"""
        return (_ptr(self.colptr), _ptr(self.rowidx), _ptr(self.values)) + self.shape


def _matrix_args(data):
    """(leading arguments of the dense or the *_csc entry point, suffix of its name, n, C, the object that
    owns the memory those arguments point into)"""
    if is_sparse(data):
        m = CSC(data)
        return m.args(), "_csc", m.shape[0], m.shape[1], m
    data = np.asfortranarray(data, dtype=np.float64)
    if data.ndim != 2:
        raise ValueError("data must be a 2-D array (features x samples)")
    n, C = data.shape
    return (_ptr(data, _dp), n, C, n), "", n, C, data


def run_pairs(data, global_na=(), pi=None, pj=None, want_counts=False, devices=None, **opt_kw):
    """One-shot call through icikt_all_pairs / icikt_pair_list with host buffers.

    data: (n, C) array (copied to Fortran order if needed), or a scipy.sparse matrix (-> the *_csc entry
    points; entries not stored are 0.0).  Returns a dict of NumPy arrays in
    pair order: raw, pvalue, taumax, completeness, status, [counts], max_taumax, timings.
    devices: list of CUDA ordinals -> icikt_all_pairs_multi (all pairs only): every device takes a
    contiguous slice of the pair order.
    """
    if devices is not None and (opt_kw.get("pair_lo", 0) or opt_kw.get("pair_hi", 0)):
        # icikt_all_pairs_multi ignores the slice and writes every pair: buffers sized for the slice would overflow
        raise ValueError("pair_lo / pair_hi select a slice on one device: over several devices run_pairs covers "
                         "all pairs")
    L = load()
    lead, sfx, n, C, keep_alive = _matrix_args(data)
    o = make_opts(want_counts=want_counts, **opt_kw)
    if pi is None:
        ptot = C * (C - 1) // 2 + (C if o.include_diag else 0)
        lo, hi = o.pair_lo, o.pair_hi
        P = ptot if (lo == 0 and hi == 0) else hi - lo
    else:
        pi = np.ascontiguousarray(pi, dtype=np.int32)
        pj = np.ascontiguousarray(pj, dtype=np.int32)
        P = int(pi.size)
    # the five result arrays are views of one allocation: one address lookup instead of five
    P = max(P, 0)
    buf = np.empty(4 * P + (P + 1) // 2, dtype=np.float64)
    raw, pv, tm, comp = buf[:P], buf[P:2 * P], buf[2 * P:3 * P], buf[3 * P:4 * P]
    status = buf[4 * P:].view(np.int32)[:P]
    counts = np.empty((P, NCOUNTS), dtype=np.int64) if want_counts else None
    a_raw = _ptr(buf)
    a_pv, a_tm, a_comp, a_status = a_raw + 8 * P, a_raw + 16 * P, a_raw + 24 * P, a_raw + 32 * P
    mx = ctypes.c_double(float("nan"))
    t = Timings()
    g, gp, ng = _global_na_array(global_na)
    if pi is None and devices is not None:
        dev = np.ascontiguousarray(list(devices), dtype=np.int32)
        rc = getattr(L, "icikt_all_pairs_multi" + sfx)(*lead, gp, ng, ctypes.byref(o), _ptr(dev, _ip),
                                                       int(dev.size), a_raw, a_pv, a_tm, a_comp, a_status,
                                                       _ptr(counts, _lp), ctypes.byref(mx), ctypes.byref(t))
    elif pi is None:
        rc = getattr(L, "icikt_all_pairs" + sfx)(*lead, gp, ng, ctypes.byref(o), a_raw, a_pv, a_tm, a_comp,
                                                 a_status, _ptr(counts, _lp), ctypes.byref(mx), ctypes.byref(t))
    else:
        rc = getattr(L, "icikt_pair_list" + sfx)(*lead, gp, ng, _ptr(pi, _ip), _ptr(pj, _ip), P,
                                                 ctypes.byref(o), a_raw, a_pv, a_tm, a_comp, a_status,
                                                 _ptr(counts, _lp), ctypes.byref(mx), ctypes.byref(t))
    check(rc)
    out = dict(raw=raw, pvalue=pv, taumax=tm, completeness=comp, status=status,
               max_taumax=mx.value, timings=t.as_dict())
    if want_counts:
        out["counts"] = counts
    return out


EDGE_NAMES = ("cor", "raw", "pvalue", "taumax", "completeness")


def _bound(v):
    return float("nan") if v is None else float(v)


def _devices_args(devices):
    """(suffix of the entry point, its (devices, n_devices) arguments, the array that owns them): the single-device
    call for devices None, otherwise its _multi twin"""
    if devices is None:
        return "", (), None
    dev = np.ascontiguousarray(list(devices), dtype=np.int32)
    return "_multi", (_ptr(dev, _ip), int(dev.size)), dev


def padj_method(p_adjust):
    """ICIKT_PADJ_* of one of R's p.adjust method names; ValueError for "hommel" and unknown names"""
    if p_adjust not in PADJ:
        raise ValueError(f"`p_adjust` must be one of {sorted(PADJ)} (hommel is not offered), got {p_adjust!r}")
    return PADJ[p_adjust]


def p_adjust(p, method, device=0):
    """R's p.adjust(p, method) on the device (icikt_p_adjust), bit for bit: NaN entries are not part of the family
    and stay NaN, and fewer than two non-NaN values leave p unchanged.  method: "bonferroni", "holm", "hochberg",
    "BH" (alias "fdr") or "BY".  Returns a float64 array of p's shape."""
    code = padj_method(method)
    L = load()
    a = np.ascontiguousarray(p, dtype=np.float64)
    out = np.empty_like(a)
    nt = ctypes.c_int64(0)
    check(L.icikt_p_adjust(_ptr(a), a.size, code, int(device), _ptr(out), ctypes.byref(nt)))
    return out


def _padj_args(p_adjust, max_padj):
    """the icikt_padj_filter of run_edges / run_cross_edges, or None without p_adjust"""
    if p_adjust is None:
        if max_padj is not None:
            raise ValueError("`max_padj` bounds the adjusted p-value: give `p_adjust` too")
        return None
    return PadjFilter(padj_method(p_adjust), 0, _bound(max_padj))


def _input(a):
    """(icikt_input of one matrix, n, C, the object that owns the memory it points into)"""
    if is_sparse(a):
        m = CSC(a)
        return Input(m.shape[1], None, 0, _ptr(m.colptr), _ptr(m.rowidx), _ptr(m.values)), m.shape[0], m.shape[1], m
    m = np.asfortranarray(a, dtype=np.float64)
    if m.ndim != 2:
        raise ValueError("x and y must be 2-D arrays (features x samples)")
    return Input(m.shape[1], _ptr(m), m.shape[0], None, None, None), m.shape[0], m.shape[1], m


def _edges_out(L, h, adjusted):
    """the rows of an icikt_edges result as a dict of arrays (with padj and n_tests from a _padj call); frees h"""
    try:
        m = int(L.icikt_edges_count(h))
        out = dict(i=np.empty(m, dtype=np.int32), j=np.empty(m, dtype=np.int32))
        out.update((k, np.empty(m, dtype=np.float64)) for k in EDGE_NAMES)
        check(L.icikt_edges_copy(h, _ptr(out["i"]), _ptr(out["j"]), *(_ptr(out[k]) for k in EDGE_NAMES)))
        if adjusted:
            out["padj"] = np.empty(m, dtype=np.float64)
            check(L.icikt_edges_copy_padj(h, _ptr(out["padj"])))
            out["n_tests"] = int(L.icikt_edges_n_tests(h))
    finally:
        L.icikt_edges_free(h)
    return out


def run_edges(data, global_na=(), min_abs_cor=None, max_pvalue=None, scale_max=True, max_edges=0, devices=None,
              p_adjust=None, max_padj=None, **opt_kw):
    """icikt_all_pairs_edges: all pairs, filtered on the device, as a long table of the pairs that pass.

    A pair is kept iff it is not degenerate, abs(cor) >= min_abs_cor and pvalue <= max_pvalue (a bound of None is
    no condition), with cor = raw / max(taumax over all pairs) if scale_max else raw.  Rows are in the pair order
    of run_pairs, and every field is bit for bit run_pairs' for that pair.  data may be a scipy.sparse matrix
    (-> icikt_all_pairs_edges_csc).  max_edges > 0 raises IciktError(ERR_LIMIT) when more pairs pass.
    devices: list of CUDA ordinals -> icikt_all_pairs_edges_multi(_csc): every device walks a contiguous slice of the
    pair order; the result is bit for bit the single-device one.
    p_adjust: one of R's p.adjust methods ("bonferroni", "holm", "hochberg", "BH" or "fdr", "BY") ->
    icikt_all_pairs_edges_padj(_multi): rows also get padj, bit for bit p.adjust(p_all, p_adjust) over the non-NaN
    p-values of every pair (p_all: run_pairs' pvalue), and the dict gets n_tests (their number); max_padj keeps the
    rows with padj <= max_padj (None: no condition) and needs p_adjust.
    Returns a dict of NumPy arrays i, j (int32), cor, raw, pvalue, taumax, completeness, plus max_taumax and
    timings."""
    adj = _padj_args(p_adjust, max_padj)
    L = load()
    msfx, dargs, dev = _devices_args(devices)
    o = make_opts(**opt_kw)
    f = EdgeFilter(_bound(min_abs_cor), _bound(max_pvalue), int(bool(scale_max)), 0, int(max_edges))
    h = ctypes.c_void_p()
    mx = ctypes.c_double(float("nan"))
    t = Timings()
    g, gp, ng = _global_na_array(global_na)
    if adj is None:
        lead, sfx, n, C, keep_alive = _matrix_args(data)
        check(getattr(L, "icikt_all_pairs_edges" + msfx + sfx)(*lead, gp, ng, ctypes.byref(o), *dargs, ctypes.byref(f),
                                                               ctypes.byref(h), ctypes.byref(mx), ctypes.byref(t)))
    else:
        xi, n, C, keep_alive = _input(data)
        check(getattr(L, "icikt_all_pairs_edges_padj" + msfx)(ctypes.byref(xi), n, gp, ng, ctypes.byref(o), *dargs,
                                                              ctypes.byref(f), ctypes.byref(adj), ctypes.byref(h),
                                                              ctypes.byref(mx), ctypes.byref(t)))
    out = _edges_out(L, h, adj is not None)
    out.update(max_taumax=mx.value, timings=t.as_dict())
    return out


def run_topk(data, global_na=(), k=10, by="abs", scale_max=True, devices=None, **opt_kw):
    """icikt_all_pairs_topk: every column's k best partners over all pairs, selected on the device.

    The candidates of column c are the columns d != c whose pair is not degenerate, ranked by abs(raw) (by="abs")
    or raw (by="signed") descending, then d ascending; column c keeps its first min(k, #candidates), best first.
    Every field is bit for bit run_pairs' for that pair, cor = raw / max_taumax if scale_max else raw.  data may be
    a scipy.sparse matrix (-> icikt_all_pairs_topk_csc).  devices: list of CUDA ordinals ->
    icikt_all_pairs_topk_multi(_csc): every device walks a contiguous slice of the pair order and the devices merge
    their lists, bit for bit the single-device result.  Returns a dict with index (C, k) int32 (-1 where
    unused), cor, raw, pvalue, taumax, completeness (C, k) float64 (NaN where unused), n_neighbors (C,) int32,
    max_taumax and timings."""
    if by not in TOPK_BY:
        raise ValueError(f"by must be one of {sorted(TOPK_BY)}")
    L = load()
    lead, sfx, n, C, keep_alive = _matrix_args(data)
    msfx, dargs, dev = _devices_args(devices)
    o = make_opts(**opt_kw)
    k = int(k)
    kk = k if 1 <= k <= TOPK_MAX else 0  # a k the library refuses gets no arrays
    k = k if -2 ** 31 <= k < 2 ** 31 else 0  # and reaches it as a refused int32
    out = dict(index=np.empty((C, kk), dtype=np.int32))
    out.update((name, np.empty((C, kk), dtype=np.float64)) for name in EDGE_NAMES)
    out["n_neighbors"] = np.empty(C, dtype=np.int32)
    mx = ctypes.c_double(float("nan"))
    t = Timings()
    g, gp, ng = _global_na_array(global_na)
    check(getattr(L, "icikt_all_pairs_topk" + msfx + sfx)(*lead, gp, ng, ctypes.byref(o), *dargs, k, TOPK_BY[by],
                                                          int(bool(scale_max)), _ptr(out["index"]),
                                                          _ptr(out["n_neighbors"]),
                                                          *(_ptr(out[name]) for name in EDGE_NAMES), ctypes.byref(mx),
                                                          ctypes.byref(t)))
    out.update(max_taumax=mx.value, timings=t.as_dict())
    return out


def _cross_inputs(x, y):
    """(icikt_input of x, of y, n, Cx, Cy, the objects that own the memory they point into) for the cross calls; x
    and y may each be a NumPy array or a scipy.sparse matrix"""
    ins, keep = [], []
    for a in (x, y):
        i, n, c, m = _input(a)
        ins.append(i)
        keep.append((m, (n, c)))
    (_, (nx, cx)), (_, (ny, cy)) = keep
    if nx != ny:
        raise ValueError(f"x has {nx} rows and y has {ny}: the cross calls need the same rows")
    return ins[0], ins[1], nx, cx, cy, keep


def run_cross(x, y, global_na=(), devices=None, **opt_kw):
    """icikt_cross_pairs: every column of x against every column of y (same rows), pair p = i * Cy + j in x-major
    order; pair_lo / pair_hi select a slice (0, 0: all).  Every field is bit for bit run_pairs(hstack([x, y]),
    pi=i, pj=Cx + j)'s.  x and y may each be a NumPy array or a scipy.sparse matrix.  devices: list of CUDA
    ordinals -> icikt_cross_pairs_multi: every device computes a contiguous slice of the pairs; the result is bit for
    bit the single-device one.  Returns a dict of NumPy arrays in pair order: raw, pvalue, taumax, completeness,
    status, plus max_taumax and timings."""
    L = load()
    xi, yi, n, cx, cy, keep_alive = _cross_inputs(x, y)
    msfx, dargs, dev = _devices_args(devices)
    o = make_opts(**opt_kw)
    P = cx * cy if (o.pair_lo == 0 and o.pair_hi == 0) else max(o.pair_hi - o.pair_lo, 0)
    buf = np.empty(4 * P + (P + 1) // 2, dtype=np.float64)
    raw, pv, tm, comp = buf[:P], buf[P:2 * P], buf[2 * P:3 * P], buf[3 * P:4 * P]
    status = buf[4 * P:].view(np.int32)[:P]
    a = _ptr(buf)
    mx = ctypes.c_double(float("nan"))
    t = Timings()
    g, gp, ng = _global_na_array(global_na)
    check(getattr(L, "icikt_cross_pairs" + msfx)(ctypes.byref(xi), ctypes.byref(yi), n, gp, ng, ctypes.byref(o),
                                                 *dargs, a, a + 8 * P, a + 16 * P, a + 24 * P, a + 32 * P,
                                                 ctypes.byref(mx), ctypes.byref(t)))
    return dict(raw=raw, pvalue=pv, taumax=tm, completeness=comp, status=status, max_taumax=mx.value,
                timings=t.as_dict())


def run_cross_edges(x, y, global_na=(), min_abs_cor=None, max_pvalue=None, scale_max=True, max_edges=0, devices=None,
                    p_adjust=None, max_padj=None, **opt_kw):
    """icikt_cross_edges: the pairs of x's columns with y's columns that pass the filter of run_edges, in cross
    order, filtered on the device.  devices: list of CUDA ordinals -> icikt_cross_edges_multi, bit for bit the
    single-device result.  p_adjust / max_padj as in run_edges (-> icikt_cross_edges_padj(_multi)), the family being
    every pair of the cross order.  Returns the dict of run_edges; i indexes x's columns, j y's."""
    adj = _padj_args(p_adjust, max_padj)
    L = load()
    xi, yi, n, cx, cy, keep_alive = _cross_inputs(x, y)
    msfx, dargs, dev = _devices_args(devices)
    o = make_opts(**opt_kw)
    f = EdgeFilter(_bound(min_abs_cor), _bound(max_pvalue), int(bool(scale_max)), 0, int(max_edges))
    h = ctypes.c_void_p()
    mx = ctypes.c_double(float("nan"))
    t = Timings()
    g, gp, ng = _global_na_array(global_na)
    if adj is None:
        check(getattr(L, "icikt_cross_edges" + msfx)(ctypes.byref(xi), ctypes.byref(yi), n, gp, ng, ctypes.byref(o),
                                                     *dargs, ctypes.byref(f), ctypes.byref(h), ctypes.byref(mx),
                                                     ctypes.byref(t)))
    else:
        check(getattr(L, "icikt_cross_edges_padj" + msfx)(ctypes.byref(xi), ctypes.byref(yi), n, gp, ng,
                                                          ctypes.byref(o), *dargs, ctypes.byref(f), ctypes.byref(adj),
                                                          ctypes.byref(h), ctypes.byref(mx), ctypes.byref(t)))
    out = _edges_out(L, h, adj is not None)
    out.update(max_taumax=mx.value, timings=t.as_dict())
    return out


def _count_filters(filters):
    """the icikt_edge_filter array of an edge-count call from a sequence of (min_abs_cor, max_pvalue), None as no
    bound; an empty or too long list reaches the library as it is and is refused there"""
    fl = [(None, None) if f is None else tuple(f) for f in filters]
    if any(len(f) != 2 for f in fl):
        raise ValueError("every filter is a pair (min_abs_cor, max_pvalue), None as no bound")
    arr = (EdgeFilter * max(len(fl), 1))()
    for k, (t, a) in enumerate(fl):
        arr[k] = EdgeFilter(_bound(t), _bound(a), 0, 0, 0)
    return arr, len(fl)


def run_count_edges(data, global_na=(), filters=((None, None),), devices=None, want_degree=True, **opt_kw):
    """icikt_all_pairs_count_edges: for every filter (min_abs_cor, max_pvalue) of `filters` (None: no bound), the
    number of pairs that pass it -- exactly the rows run_edges(..., scale_max=False) returns with that filter -- and
    every column's degree among them, in one walk of the pair order; no pair comes back.  data may be a scipy.sparse
    matrix.  devices: list of CUDA ordinals -> icikt_all_pairs_count_edges_multi, bit for bit the single-device
    result.  Returns a dict with n_pass (T,) int64, degree (C, T) int64 (a diagonal pair counts once; None without
    want_degree), status_counts (NSTATUS,) int64 (pairs per status class), max_taumax and timings."""
    L = load()
    arr, T = _count_filters(filters)
    xi, n, C, keep_alive = _input(data)
    msfx, dargs, dev = _devices_args(devices)
    o = make_opts(**opt_kw)
    n_pass = np.zeros(max(T, 1), dtype=np.int64)
    degree = np.zeros((C, max(T, 1)), dtype=np.int64) if want_degree else None
    hist = np.zeros(NSTATUS, dtype=np.int64)
    mx = ctypes.c_double(float("nan"))
    t = Timings()
    g, gp, ng = _global_na_array(global_na)
    check(getattr(L, "icikt_all_pairs_count_edges" + msfx)(ctypes.byref(xi), n, gp, ng, ctypes.byref(o), *dargs, arr,
                                                           T, _ptr(n_pass), _ptr(degree), _ptr(hist), ctypes.byref(mx),
                                                           ctypes.byref(t)))
    return dict(n_pass=n_pass, degree=degree, status_counts=hist, max_taumax=mx.value, timings=t.as_dict())


def run_cross_count_edges(x, y, global_na=(), filters=((None, None),), devices=None, want_degree=True, **opt_kw):
    """icikt_cross_count_edges: run_count_edges over the cross order of x against y (the rows run_cross_edges(...,
    scale_max=False) returns).  devices -> icikt_cross_count_edges_multi, bit for bit the single-device result.
    Returns a dict with n_pass (T,), x_degree (Cx, T), y_degree (Cy, T) (None without want_degree), status_counts,
    max_taumax and timings."""
    L = load()
    arr, T = _count_filters(filters)
    xi, yi, n, cx, cy, keep_alive = _cross_inputs(x, y)
    msfx, dargs, dev = _devices_args(devices)
    o = make_opts(**opt_kw)
    n_pass = np.zeros(max(T, 1), dtype=np.int64)
    xd = np.zeros((cx, max(T, 1)), dtype=np.int64) if want_degree else None
    yd = np.zeros((cy, max(T, 1)), dtype=np.int64) if want_degree else None
    hist = np.zeros(NSTATUS, dtype=np.int64)
    mx = ctypes.c_double(float("nan"))
    t = Timings()
    g, gp, ng = _global_na_array(global_na)
    check(getattr(L, "icikt_cross_count_edges" + msfx)(ctypes.byref(xi), ctypes.byref(yi), n, gp, ng, ctypes.byref(o),
                                                       *dargs, arr, T, _ptr(n_pass), _ptr(xd), _ptr(yd), _ptr(hist),
                                                       ctypes.byref(mx), ctypes.byref(t)))
    return dict(n_pass=n_pass, x_degree=xd, y_degree=yd, status_counts=hist, max_taumax=mx.value,
                timings=t.as_dict())


CROSS_SIDES = {"x": (True, False), "y": (False, True), "both": (True, True)}


def run_cross_topk(x, y, global_na=(), k=10, by="abs", scale_max=True, side="both", devices=None, **opt_kw):
    """icikt_cross_topk: each column's k best partners in the other matrix, in the order of run_topk.  side "x": the
    lists of x's columns (partners are y indices), "y": of y's columns (partners are x indices), "both".  devices:
    list of CUDA ordinals -> icikt_cross_topk_multi: every device walks a contiguous slice of the pairs and the
    devices merge their lists, bit for bit the single-device result.  Returns a dict with x_side and/or y_side (each
    the per-column arrays of run_topk: index, n_neighbors, cor, raw, pvalue, taumax, completeness), max_taumax and
    timings."""
    if by not in TOPK_BY:
        raise ValueError(f"by must be one of {sorted(TOPK_BY)}")
    if side not in CROSS_SIDES:
        raise ValueError(f"side must be one of {sorted(CROSS_SIDES)}")
    L = load()
    xi, yi, n, cx, cy, keep_alive = _cross_inputs(x, y)
    msfx, dargs, dev = _devices_args(devices)
    o = make_opts(**opt_kw)
    k = int(k)
    kk = k if 1 <= k <= TOPK_MAX else 0  # a k the library refuses gets no arrays
    k = k if -2 ** 31 <= k < 2 ** 31 else 0  # and reaches it as a refused int32
    out, lists = {}, []
    for name, want, C in (("x_side", CROSS_SIDES[side][0], cx), ("y_side", CROSS_SIDES[side][1], cy)):
        if not want:
            lists.append(None)
            continue
        d = dict(index=np.empty((C, kk), dtype=np.int32), n_neighbors=np.empty(C, dtype=np.int32))
        d.update((f, np.empty((C, kk), dtype=np.float64)) for f in EDGE_NAMES)
        out[name] = d
        lists.append(TopkLists(_ptr(d["index"]), _ptr(d["n_neighbors"]), *(_ptr(d[f]) for f in EDGE_NAMES)))
    mx = ctypes.c_double(float("nan"))
    t = Timings()
    g, gp, ng = _global_na_array(global_na)
    check(getattr(L, "icikt_cross_topk" + msfx)(ctypes.byref(xi), ctypes.byref(yi), n, gp, ng, ctypes.byref(o),
                                                *dargs, k, TOPK_BY[by], int(bool(scale_max)),
                                                *(ctypes.byref(v) if v is not None else None for v in lists),
                                                ctypes.byref(mx), ctypes.byref(t)))
    out.update(max_taumax=mx.value, timings=t.as_dict())
    return out


MATRIX_NAMES = ("cor", "raw", "pvalue", "taumax", "completeness")


def run_matrices(data, global_na=(), scale_max=True, diag_good=True, n_good=None, pi=None, pj=None,
                 want=MATRIX_NAMES, devices=None, **opt_kw):
    """icikt_matrices: the pair results as symmetric C x C matrices filled on the device
    (scale_and_reshape, R/kendalltau.R:357-421).  Returns the requested matrices plus
    status_counts (pairs per status class), max_taumax and timings.
    devices: list of CUDA ordinals -> icikt_matrices_multi (all pairs only): the pair order is sliced
    over the devices and every device returns its own block of columns of each matrix.
    data may be a scipy.sparse matrix (-> the *_csc entry points)."""
    L = load()
    lead, sfx, n, C, keep_alive = _matrix_args(data)
    o = make_opts(**opt_kw)
    mats = {k: (np.empty((C, C), dtype=np.float64, order="F") if k in want else None) for k in MATRIX_NAMES}
    hist = np.zeros(NSTATUS, dtype=np.int64)
    mx = ctypes.c_double(float("nan"))
    t = Timings()
    g, gp, ng = _global_na_array(global_na)
    if pi is not None:
        pi = np.ascontiguousarray(pi, dtype=np.int32)
        pj = np.ascontiguousarray(pj, dtype=np.int32)
    ngood = None if n_good is None else np.ascontiguousarray(n_good, dtype=np.int32)
    if devices is not None:
        if pi is not None:
            raise ValueError("several devices: all pairs only")
        dev = np.ascontiguousarray(list(devices), dtype=np.int32)
        check(getattr(L, "icikt_matrices_multi" + sfx)(*lead, gp, ng, ctypes.byref(o), _ptr(dev, _ip), int(dev.size),
                                     int(bool(scale_max)), int(bool(diag_good)), _ptr(ngood, _ip),
                                     *(_ptr(mats[k], _dp) for k in MATRIX_NAMES), _ptr(hist, _lp), ctypes.byref(mx),
                                     ctypes.byref(t)))
        out = {k: v for k, v in mats.items() if v is not None}
        out.update(status_counts=hist, max_taumax=mx.value, timings=t.as_dict())
        return out
    check(getattr(L, "icikt_matrices" + sfx)(*lead, gp, ng, _ptr(pi, _ip), _ptr(pj, _ip),
                           0 if pi is None else int(pi.size), ctypes.byref(o), int(bool(scale_max)),
                           int(bool(diag_good)), _ptr(ngood, _ip), *(_ptr(mats[k], _dp) for k in MATRIX_NAMES),
                           _ptr(hist, _lp), ctypes.byref(mx), ctypes.byref(t)))
    out = {k: v for k, v in mats.items() if v is not None}
    out.update(status_counts=hist, max_taumax=mx.value, timings=t.as_dict())
    return out


def pairwise_completeness(data, global_na=(), pi=None, pj=None, want_matrix=False, want_pairs=True, device=0):
    """icikt_pairwise_completeness: rows missing in either column and 1 - missing/n per pair
    (all pairs in combn order followed by the diagonal when pi is None).  data may be a scipy.sparse
    matrix (-> icikt_pairwise_completeness_csc)."""
    L = load()
    lead, sfx, n, C, keep_alive = _matrix_args(data)
    if pi is not None:
        pi = np.ascontiguousarray(pi, dtype=np.int32)
        pj = np.ascontiguousarray(pj, dtype=np.int32)
        P = int(pi.size)
    else:
        P = C * (C - 1) // 2 + C
    missing = np.empty(P, dtype=np.int32) if want_pairs else None
    comp = np.empty(P, dtype=np.float64) if want_pairs else None
    mat = np.empty((C, C), dtype=np.float64, order="F") if want_matrix else None
    g, gp, ng = _global_na_array(global_na)
    check(getattr(L, "icikt_pairwise_completeness" + sfx)(*lead, gp, ng, int(device), _ptr(pi, _ip), _ptr(pj, _ip),
                                                        P, _ptr(missing, _ip), _ptr(comp, _dp), _ptr(mat, _dp)))
    out = dict(missing=missing, completeness=comp) if want_pairs else {}
    if want_matrix:
        out["matrix"] = mat
    return out


class Plan:
    """Thin RAII wrapper of the plan API (device-resident matrix, tables and results)."""

    def __init__(self, n, C, pi=None, pj=None, **opt_kw):
        self._L = load()
        self._h = ctypes.c_void_p()
        self.opts = make_opts(**opt_kw)
        if pi is not None:
            self._pi = np.ascontiguousarray(pi, dtype=np.int32)
            self._pj = np.ascontiguousarray(pj, dtype=np.int32)
            check(self._L.icikt_plan_create(ctypes.byref(self._h), n, C, _ptr(self._pi, _ip),
                                            _ptr(self._pj, _ip), self._pi.size, ctypes.byref(self.opts)))
        else:
            check(self._L.icikt_plan_create(ctypes.byref(self._h), n, C, None, None, 0,
                                            ctypes.byref(self.opts)))
        self.n, self.C = n, C
        self.P = int(self._L.icikt_plan_num_pairs(self._h))

    def upload(self, data):
        data = np.asfortranarray(data, dtype=np.float64)
        assert data.shape == (self.n, self.C)
        check(self._L.icikt_plan_upload(self._h, _ptr(data, _dp), self.n))
        self.sync()  # the host array may go away

    def set_device_matrix(self, data_ptr, ld):
        check(self._L.icikt_plan_set_device_matrix(self._h, ctypes.c_void_p(int(data_ptr)), int(ld)))

    def columns(self, global_na=()):
        g, gp, ng = _global_na_array(global_na)
        check(self._L.icikt_plan_columns(self._h, gp, ng))

    # ---- sharded K1 (one rank per GPU): upload + preprocess a slice of the columns, exchange the
    # table slices (sharding.exchange_tables), then columns_finish() releases pairs()
    def upload_columns(self, data, col_lo, col_hi):
        """`data` is the whole (n, C) Fortran-ordered host matrix; only the slice is copied."""
        assert data.flags["F_CONTIGUOUS"] and data.dtype == np.float64 and data.shape == (self.n, self.C)
        check(self._L.icikt_plan_upload_columns(self._h, _ptr(data, _dp), self.n, int(col_lo), int(col_hi)))

    def columns_range(self, global_na, col_lo, col_hi):
        g, gp, ng = _global_na_array(global_na)
        check(self._L.icikt_plan_columns_range(self._h, gp, ng, int(col_lo), int(col_hi)))

    def tables(self):
        """[(device pointer of column 0, bytes per column)] of the per-column tables to exchange."""
        arr = (Table * MAX_TABLES)()
        n = self._L.icikt_plan_tables(self._h, arr, MAX_TABLES)
        if n < 0:
            check(n)
        return [(int(arr[k].ptr), int(arr[k].bytes_per_column)) for k in range(n)]

    def columns_finish(self):
        check(self._L.icikt_plan_columns_finish(self._h))

    def pairs(self):
        check(self._L.icikt_plan_pairs(self._h))

    def sync(self):
        check(self._L.icikt_plan_sync(self._h))

    def stream(self):
        return int(self._L.icikt_plan_stream(self._h) or 0)

    def download(self, want_counts=False):
        P = self.P
        raw, pv, tm, comp = (np.empty(P, dtype=np.float64) for _ in range(4))
        status = np.empty(P, dtype=np.int32)
        counts = np.empty((P, NCOUNTS), dtype=np.int64) if want_counts else None
        mx = ctypes.c_double(float("nan"))
        check(self._L.icikt_plan_download(self._h, _ptr(raw, _dp), _ptr(pv, _dp), _ptr(tm, _dp),
                                          _ptr(comp, _dp), _ptr(status, _ip), _ptr(counts, _lp),
                                          ctypes.byref(mx)))
        out = dict(raw=raw, pvalue=pv, taumax=tm, completeness=comp, status=status, max_taumax=mx.value)
        if want_counts:
            out["counts"] = counts
        return out

    def column_n_na(self):
        a = np.empty(self.C, dtype=np.int32)
        check(self._L.icikt_plan_column_info(self._h, _ptr(a, _ip)))
        return a

    def timings(self):
        t = Timings()
        check(self._L.icikt_plan_timings(self._h, ctypes.byref(t)))
        return t.as_dict()

    def close(self):
        if self._h:
            self._L.icikt_plan_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def pnorm_device(z, lower_tail=True, device=0):
    z = np.ascontiguousarray(z, dtype=np.float64)
    out = np.empty_like(z)
    check(load().icikt_pnorm_device(_ptr(z, _dp), z.size, int(bool(lower_tail)), _ptr(out, _dp), device))
    return out


def release_workspace():
    load().icikt_release_workspace()


def measure_smem_bandwidth(device=0):
    """(GB/s with 32-bit accesses, GB/s with 128-bit accesses) of a conflict-free load+store sweep."""
    a, b = ctypes.c_double(0), ctypes.c_double(0)
    check(load().icikt_measure_smem_bandwidth(device, ctypes.byref(a), ctypes.byref(b)))
    return a.value, b.value


def measure_issue_rate(device=0):
    """(LOP3 only, IMAD only, interleaved) sustained issue rate in G warp-instructions/s over the GPU."""
    a, f, m = ctypes.c_double(0), ctypes.c_double(0), ctypes.c_double(0)
    check(load().icikt_measure_issue_rate(device, ctypes.byref(a), ctypes.byref(f), ctypes.byref(m)))
    return a.value, f.value, m.value


def stage_table(C, include_diag=False, cta_slots=296, n_blocks=8):
    """The launches of the pipelined one-shot call for C columns (host only, no device needed):
    (units [U, 4] = slot, first column, other column of the first pair, pairs;
     launches [L, 6] = col_lo, col_hi, unit_lo, unit_hi, slot_lo, slot_hi)."""
    L = load()
    nl = ctypes.c_int64(0)
    nu = L.icikt_stage_table(C, int(bool(include_diag)), cta_slots, n_blocks, 0, None, 0, None, ctypes.byref(nl))
    if nu < 0:
        check(int(nu))
    units = np.zeros((max(nu, 1), 4), dtype=np.int64)
    launches = np.zeros((max(nl.value, 1), 6), dtype=np.int64)
    L.icikt_stage_table(C, int(bool(include_diag)), cta_slots, n_blocks, nu, units.ctypes.data, nl.value,
                        launches.ctypes.data, ctypes.byref(nl))
    return units[:nu], launches[:nl.value]


def launch_shape(n, tier=0, n_sm=148, complete_obs=False):
    """The pair kernel's launch shape for n rows (host only): dict(warps, runs, region_bytes, variant, cap, stage_rows);
    variant: 'smem' two sequence buffers in shared memory, 'inplace', 'gmem' global scratch."""
    out = np.zeros(8, dtype=np.int32)
    check(load().icikt_launch_shape(int(n), int(tier), int(n_sm), int(bool(complete_obs)), out.ctypes.data))
    return dict(warps=int(out[0]), runs=int(out[1]), region_bytes=int(out[2]),
                variant=("smem", "inplace", "gmem")[int(out[3])], cap=int(out[4]), stage_rows=int(out[5]))


def pass_a_radix(n):
    """whether pass A runs radix-16 levels at length n (host only; the same for every tier)"""
    out = np.zeros(8, dtype=np.int32)
    check(load().icikt_launch_shape(int(n), 0, 148, 0, out.ctypes.data))
    return bool(out[6])


def pair_from_index(C, index, include_diag=False):
    i, j = ctypes.c_int32(), ctypes.c_int32()
    check(load().icikt_pair_from_index(C, int(bool(include_diag)), int(index), ctypes.byref(i), ctypes.byref(j)))
    return i.value, j.value
