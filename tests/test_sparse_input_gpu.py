"""Sparse (CSC) input on the GPU: every result of a *_csc call must be the dense call's on A.toarray(), bit for
bit (NaN in the same places, with the same payload).  The lengths cover the fused, shared-memory and global
column sorts and the in-place pair kernel; the densities include an all-implicit and a fully stored column;
global_na with and without 0 and negative values put an implicit 0 below or inside the order of a column."""
import numpy as np
import pytest
import scipy.sparse as sp

import icikendalltau_b200 as ik
from icikendalltau_b200 import _lib
from tests.test_gpu_parity import assert_parity, oracle_pairs

pytestmark = pytest.mark.gpu

LENGTHS = [50, 512, 513, 8192, 8193, 22528, 22529, 60000]
DENSITIES = [0.0, 0.01, 0.3, 1.0]
NA_WITH_ZERO = (np.nan, np.inf, 0.0)
NA_WITHOUT_ZERO = (np.nan, np.inf)
PAIR_KEYS = ("raw", "pvalue", "taumax", "completeness", "status", "counts")


def make_sparse(n, C, density, seed, fmt="csc"):
    """n x C with about `density` of the entries stored: negative and positive values, ties, stored NaN, +-Inf,
    0.0 and -0.0; column 0 stores nothing, column 1 stores every row"""
    rng = np.random.default_rng(seed)
    d = rng.normal(size=(n, 1)) + 0.7 * rng.normal(size=(n, C))
    d[:, ::3] = np.round(d[:, ::3] * 4)  # ties, integer values that include 0
    stored = rng.random((n, C)) < density
    stored[:, 0] = False
    stored[:, 1] = True
    r, c = np.nonzero(stored)
    v = d[r, c]
    special = rng.random(v.size)
    v[special < 0.01] = np.nan
    v[(special >= 0.01) & (special < 0.015)] = np.inf
    v[(special >= 0.015) & (special < 0.02)] = -np.inf
    v[(special >= 0.02) & (special < 0.03)] = 0.0
    v[(special >= 0.03) & (special < 0.04)] = -0.0
    a = sp.csc_matrix((v, (r, c)), shape=(n, C))
    return a if fmt == "csc" else a.asformat(fmt)


def dense_of(a):
    return np.asfortranarray(a.toarray())


def same_bits(x, y, what):
    x, y = np.asarray(x), np.asarray(y)
    assert x.shape == y.shape and x.dtype == y.dtype, what
    if x.dtype == np.float64:
        assert np.array_equal(x.view(np.int64), y.view(np.int64)), what
    else:
        assert np.array_equal(x, y), what


def same_scalar(x, y, what):
    assert np.array_equal(np.float64(x).view(np.int64), np.float64(y).view(np.int64)), what


def same_pairs(a, b, what):
    for k in PAIR_KEYS:
        assert (k in a) == (k in b), what
        if k in a:
            same_bits(a[k], b[k], f"{what}: {k}")
    same_scalar(a["max_taumax"], b["max_taumax"], f"{what}: max_taumax")


def same_matrices(a, b, what):
    for k in _lib.MATRIX_NAMES + ("status_counts",):
        same_bits(a[k], b[k], f"{what}: {k}")
    same_scalar(a["max_taumax"], b["max_taumax"], f"{what}: max_taumax")


@pytest.mark.parametrize("n", LENGTHS)
def test_run_pairs_matches_dense(n):
    C = 10
    for di, density in enumerate(DENSITIES):
        a = make_sparse(n, C, density, seed=n + di)
        d = dense_of(a)
        for gna in (NA_WITH_ZERO, NA_WITHOUT_ZERO):
            for persp in ("global", "local", "complete"):
                if persp == "complete" and gna is NA_WITHOUT_ZERO:
                    continue
                kw = dict(perspective=persp, want_counts=True)
                what = f"n={n} density={density} global_na={gna} {persp}"
                same_pairs(ik.run_pairs(a, gna, **kw), ik.run_pairs(d, gna, **kw), what)


@pytest.mark.parametrize("n", [513, 8193, 22529])
def test_pair_list_and_matrices_match_dense(n):
    C = 9
    a = make_sparse(n, C, 0.3, seed=7 * n)
    d = dense_of(a)
    pi = np.array([0, 0, 1, 2, 3, 5, 8, 4, 4], dtype=np.int32)
    pj = np.array([1, 5, 2, 7, 3, 6, 0, 4, 8], dtype=np.int32)
    n_good = (~ik.setup_missing_matrix(d, NA_WITH_ZERO)).sum(axis=0)
    for gna in (NA_WITH_ZERO, NA_WITHOUT_ZERO):
        kw = dict(perspective="global", want_counts=True)
        same_pairs(ik.run_pairs(a, gna, pi=pi, pj=pj, **kw), ik.run_pairs(d, gna, pi=pi, pj=pj, **kw),
                   f"pair list n={n} {gna}")
        for scale_max in (True, False):
            for diag_good in (True, False):
                for ng in (None, n_good):
                    mk = dict(scale_max=scale_max, diag_good=diag_good, n_good=ng, perspective="local")
                    what = f"matrices n={n} {gna} scale_max={scale_max} diag_good={diag_good} n_good={ng is not None}"
                    same_matrices(_lib.run_matrices(a, gna, **mk), _lib.run_matrices(d, gna, **mk), what)
                    same_matrices(_lib.run_matrices(a, gna, pi=pi, pj=pj, **mk),
                                  _lib.run_matrices(d, gna, pi=pi, pj=pj, **mk), f"{what} pair list")


@pytest.mark.parametrize("n", [50, 8193, 60000])
def test_pairwise_completeness_matches_dense(n):
    C = 11
    for density in DENSITIES:
        a = make_sparse(n, C, density, seed=n + 99)
        d = dense_of(a)
        for gna in (NA_WITH_ZERO, NA_WITHOUT_ZERO, (0.0,)):
            what = f"completeness n={n} density={density} {gna}"
            x = _lib.pairwise_completeness(a, gna, want_matrix=True)
            y = _lib.pairwise_completeness(d, gna, want_matrix=True)
            for k in ("missing", "completeness", "matrix"):
                same_bits(x[k], y[k], f"{what}: {k}")
            pi, pj = np.array([3, 0, 10], dtype=np.int32), np.array([3, 1, 2], dtype=np.int32)
            x = _lib.pairwise_completeness(a, gna, pi=pi, pj=pj)
            y = _lib.pairwise_completeness(d, gna, pi=pi, pj=pj)
            for k in ("missing", "completeness"):
                same_bits(x[k], y[k], f"{what} pair list: {k}")


def test_multi_gpu_calls_match_dense():
    devices = list(range(_lib.load().icikt_device_count()))
    for n in (513, 22529):
        a = make_sparse(n, 23, 0.3, seed=n)
        d = dense_of(a)
        for gna in (NA_WITH_ZERO, NA_WITHOUT_ZERO):
            kw = dict(perspective="global", want_counts=True)
            same_pairs(_lib.run_pairs(a, gna, devices=devices, **kw), _lib.run_pairs(d, gna, devices=devices, **kw),
                       f"multi pairs n={n} {gna}")
            same_pairs(_lib.run_pairs(a, gna, devices=devices, **kw), _lib.run_pairs(d, gna, **kw),
                       f"multi pairs vs one device n={n} {gna}")
            for diag_good in (True, False):
                mk = dict(scale_max=True, diag_good=diag_good, perspective="local")
                same_matrices(_lib.run_matrices(a, gna, devices=devices, **mk),
                              _lib.run_matrices(d, gna, devices=devices, **mk), f"multi matrices n={n} {gna} {diag_good}")


def test_pipelined_call_matches_dense(monkeypatch):
    """16 500 x 256 doubles are 33.8 MB: the pipelined one-shot call runs for the dense twin and, since it is
    chosen on the dense size, for the sparse call too; at half density the stored arrays are large enough
    for the pinned-chunk upload"""
    a = make_sparse(16500, 256, 0.5, seed=5)
    d = dense_of(a)
    kw = dict(perspective="global", want_counts=True)
    _lib.release_workspace()
    piped = ik.run_pairs(a, NA_WITH_ZERO, **kw)
    same_pairs(piped, ik.run_pairs(d, NA_WITH_ZERO, **kw), "16500 x 256 pipelined")
    monkeypatch.setenv("ICIKT_NO_PIPELINE", "1")
    _lib.release_workspace()
    plain = ik.run_pairs(a, NA_WITH_ZERO, **kw)
    assert piped["timings"]["n_launches"] > plain["timings"]["n_launches"], "the pipelined path did not run"
    same_pairs(plain, piped, "16500 x 256 plain vs pipelined")
    monkeypatch.delenv("ICIKT_NO_PIPELINE")
    _lib.release_workspace()


def test_pipelined_small_case_matches_dense(monkeypatch):
    a = make_sparse(700, 260, 0.3, seed=11)
    d = dense_of(a)
    monkeypatch.setenv("ICIKT_PIPELINE_MIN_BYTES", "1")
    _lib.release_workspace()
    for gna in (NA_WITH_ZERO, NA_WITHOUT_ZERO):
        kw = dict(perspective="local", want_counts=True, include_diag=True)
        same_pairs(ik.run_pairs(a, gna, **kw), ik.run_pairs(d, gna, **kw), f"pipelined small {gna}")
        mk = dict(scale_max=True, diag_good=False, perspective="global")
        same_matrices(_lib.run_matrices(a, gna, **mk), _lib.run_matrices(d, gna, **mk), f"pipelined matrices {gna}")
    _lib.release_workspace()


def test_cached_workspace_across_input_forms():
    """the one-shot plan is cached by shape: a sparse call, a dense call of the same shape, then sparse calls
    with more and with fewer stored entries must each still give their dense twin's results"""
    n, C = 8193, 40
    _lib.release_workspace()
    kw = dict(perspective="global", want_counts=True)
    a1 = make_sparse(n, C, 0.05, seed=1)
    d1 = dense_of(a1)
    r1 = ik.run_pairs(a1, NA_WITH_ZERO, **kw)
    x = make_sparse(n, C, 0.5, seed=2)
    rd = ik.run_pairs(dense_of(x), NA_WITHOUT_ZERO, **kw)  # dense, same shape, on the cached plan
    a2 = make_sparse(n, C, 0.6, seed=3)   # more entries: the CSC buffers grow
    r2 = ik.run_pairs(a2, NA_WITHOUT_ZERO, **kw)
    a3 = make_sparse(n, C, 0.02, seed=4)  # fewer
    r3 = ik.run_pairs(a3, NA_WITH_ZERO, **kw)
    _lib.release_workspace()
    same_pairs(r1, ik.run_pairs(d1, NA_WITH_ZERO, **kw), "sparse, first call")
    _lib.release_workspace()
    same_pairs(rd, ik.run_pairs(dense_of(x), NA_WITHOUT_ZERO, **kw), "dense after sparse")
    _lib.release_workspace()
    same_pairs(r2, ik.run_pairs(dense_of(a2), NA_WITHOUT_ZERO, **kw), "sparse, more entries")
    _lib.release_workspace()
    same_pairs(r3, ik.run_pairs(dense_of(a3), NA_WITH_ZERO, **kw), "sparse, fewer entries")
    _lib.release_workspace()


def test_sparse_matches_oracle():
    """about 200 pairs of one sparse case against the CPU oracle, at the parity bars"""
    a = make_sparse(3000, 21, 0.4, seed=2024)
    d = dense_of(a)
    for gna, persp in ((NA_WITH_ZERO, "global"), (NA_WITHOUT_ZERO, "local")):
        got = ik.run_pairs(a, gna, perspective=persp, want_counts=True)
        assert got["raw"].size == 210
        assert_parity(got, oracle_pairs(d, global_na=gna, perspective=persp), f"sparse oracle {persp}")


@pytest.mark.parametrize("fmt", ["csc", "csr", "coo"])
def test_api_on_sparse_input_matches_dense(fmt):
    a = make_sparse(2000, 12, 0.3, seed=77, fmt=fmt)
    d = a.toarray()
    names = [f"s{i}" for i in range(12)]
    for kw in (dict(), dict(scale_max=False, diag_good=False), dict(include_only="s3"),
               dict(global_na=(np.nan, -1.0), perspective="local")):
        x = ik.ici_kendalltau(a, colnames=names, **kw)
        y = ik.ici_kendalltau(d, colnames=names, **kw)
        for k in _lib.MATRIX_NAMES + ("keep",):
            same_bits(x[k], y[k], f"ici_kendalltau {fmt} {kw}: {k}")
    x = ik.ici_kendalltau(a, colnames=names, return_matrix=False)["cor"]
    y = ik.ici_kendalltau(d, colnames=names, return_matrix=False)["cor"]
    for k in ("raw", "pvalue", "taumax", "completeness", "cor"):
        same_bits(x[k], y[k], f"long table {fmt}: {k}")
    n_gpus = _lib.load().icikt_device_count()
    x = ik.ici_kendalltau(a, colnames=names, n_gpus=n_gpus)
    y = ik.ici_kendalltau(d, colnames=names, n_gpus=n_gpus)
    for k in _lib.MATRIX_NAMES + ("keep",):
        same_bits(x[k], y[k], f"ici_kendalltau n_gpus={n_gpus} {fmt}: {k}")
    for kw in (dict(), dict(include_only="s1"), dict(return_matrix=False), dict(global_na=(np.nan,))):
        x = ik.pairwise_completeness(a, colnames=names, **kw)
        y = ik.pairwise_completeness(d, colnames=names, **kw)
        if isinstance(x, dict):
            for k in ("missingness", "completeness"):
                same_bits(x[k], y[k], f"pairwise_completeness {fmt} {kw}: {k}")
        else:
            same_bits(x, y, f"pairwise_completeness {fmt} {kw}")
