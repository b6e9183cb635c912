"""The filtered all-pairs call (icikt_all_pairs_edges) on the GPU.  Every comparison is bit for bit against run_pairs
on the same input, masked by the edge predicate:

    status == 0 & (t is None | abs(cor) >= t) & (a is None | pvalue <= a),  cor = raw / max_taumax or raw.

Windows of 1, 7 and 4096 pairs (ICIKT_EDGE_WINDOW) cut units and tiles mid-way; the late-maximum cases put the
largest taumax in the last window, so that earlier windows hold rows the final trim has to remove."""
import numpy as np
import pytest
import scipy.sparse as sp

import icikendalltau_b200 as ik
from icikendalltau_b200 import _lib
from tests.test_gpu_parity import gen

pytestmark = pytest.mark.gpu

T_BOUNDS = (None, 0.0, 0.1, 0.5, 1.01)
A_BOUNDS = (None, 1e-3, 1.0)
FIELDS = ("cor", "raw", "pvalue", "taumax", "completeness")


def pair_order(C, include_diag):
    iu = np.triu_indices(C, 1)
    pi, pj = iu[0].astype(np.int32), iu[1].astype(np.int32)
    if include_diag:
        d = np.arange(C, dtype=np.int32)
        pi, pj = np.concatenate([pi, d]), np.concatenate([pj, d])
    return pi, pj


def expected(full, C, t, a, scale_max, include_diag=False):
    """the per-pair result of run_pairs, masked by the edge predicate"""
    pi, pj = pair_order(C, include_diag)
    raw, pv = full["raw"], full["pvalue"]
    cor = raw / full["max_taumax"] if scale_max else raw
    sel = full["status"] == 0
    with np.errstate(invalid="ignore"):
        if t is not None:
            sel &= np.abs(cor) >= t
        if a is not None:
            sel &= pv <= a
    out = dict(i=pi[sel], j=pj[sel], cor=cor[sel])
    out.update((k, full[k][sel]) for k in ("raw", "pvalue", "taumax", "completeness"))
    return out


def same(got, want, what):
    for k in ("i", "j") + FIELDS:
        g, w = np.asarray(got[k]), np.asarray(want[k])
        assert g.dtype == w.dtype and g.shape == w.shape, f"{what}: {k} {g.dtype}{g.shape} vs {w.dtype}{w.shape}"
        if g.dtype == np.float64:
            assert np.array_equal(g.view(np.int64), w.view(np.int64)), f"{what}: {k}"
        else:
            assert np.array_equal(g, w), f"{what}: {k}"


def same_max(got, full, what):
    assert np.array_equal(np.float64(got["max_taumax"]).view(np.int64), np.float64(full["max_taumax"]).view(np.int64)), what


def check_grid(x, persp, what, gna=(), ts=T_BOUNDS, As=A_BOUNDS, include_diag=False):
    C = x.shape[1]
    full = ik.run_pairs(x, gna, perspective=persp, include_diag=include_diag)
    for scale_max in (True, False):
        for t in ts:
            for a in As:
                got = ik.run_edges(x, gna, min_abs_cor=t, max_pvalue=a, scale_max=scale_max, perspective=persp,
                                   include_diag=include_diag)
                w = f"{what} {persp} scale_max={scale_max} t={t} a={a}"
                same(got, expected(full, C, t, a, scale_max, include_diag), w)
                same_max(got, full, w)
    return full


SHAPES = [(2000, 300), (5000, 120), (20000, 64), (60000, 24)]  # the last one runs the in-place pair kernel


@pytest.mark.parametrize("n,C", SHAPES)
@pytest.mark.parametrize("kind", ["normal", "mixed", "ties"])
def test_edges_equal_masked_pairs(n, C, kind):
    x = gen(n, C, kind, 0.1, seed=n + C)
    for persp in ("global", "local"):
        check_grid(x, persp, f"{n}x{C} {kind}")
    if n == 60000:
        assert _lib.launch_shape(n)["variant"] == "inplace"


@pytest.mark.parametrize("window", [1, 7, 4096])
def test_small_windows(monkeypatch, window):
    """windows that cut units and tiles mid-way; window 1 on a small matrix (one pair per window)"""
    monkeypatch.setenv("ICIKT_EDGE_WINDOW", str(window))
    n, C = (300, 30) if window == 1 else (2000, 120)
    x = gen(n, C, "mixed", 0.15, seed=window)
    check_grid(x, "global", f"window={window}", ts=(None, 0.0, 0.3), As=(None, 1e-3), include_diag=window == 7)
    check_grid(x, "local", f"window={window}", ts=(0.5,), As=(None,))


def late_maximum_matrix(n, C, seed, all_missing=False):
    """every column has missing values except the last two: the pair with the largest taumax is the last pair of
    the triangle.  all_missing: the last two lose a row too, so M < 1."""
    rng = np.random.default_rng(seed)
    x = rng.normal(size=(n, 1)) + rng.normal(size=(n, C))
    for c in range(C - (0 if all_missing else 2)):
        x[rng.random(n) < rng.uniform(0.2, 0.5), c] = np.nan
    if all_missing:
        x[0, C - 2] = x[1, C - 1] = np.nan
    return np.asfortranarray(x)


@pytest.mark.parametrize("window", [7, 4096, None])
def test_late_maximum(monkeypatch, window):
    if window:
        monkeypatch.setenv("ICIKT_EDGE_WINDOW", str(window))
    n, C = 1500, 100
    x = late_maximum_matrix(n, C, seed=3)
    for persp in ("global", "local"):
        full = ik.run_pairs(x, (), perspective=persp)
        tm = full["taumax"]
        assert np.nanargmax(tm) == tm.size - 1 and tm[-1] == 1.0  # the maximum comes last
        M_early = np.nanmax(tm[:-1])
        t = float(np.quantile(np.abs(full["raw"][full["status"] == 0]), 0.9))
        # rows the running maximum keeps but the final one removes exist
        early = (full["status"] == 0) & (np.abs(full["raw"]) >= t * M_early) & (np.abs(full["raw"] / tm[-1]) < t)
        assert early.sum() > 0
        for a in (None, 1e-3):
            got = ik.run_edges(x, (), min_abs_cor=t, max_pvalue=a, perspective=persp)
            same(got, expected(full, C, t, a, True), f"late maximum {persp} window={window} a={a}")
            same_max(got, full, "late maximum")


def test_maximum_below_one():
    x = late_maximum_matrix(1500, 60, seed=4, all_missing=True)
    for persp in ("global", "local"):
        full = check_grid(x, persp, "M < 1", ts=(0.3, 0.5, 0.9), As=(None,))
        assert full["max_taumax"] < 1.0


def test_degenerate_pairs_never_appear():
    rng = np.random.default_rng(5)
    x = rng.normal(size=(500, 12))
    x[:, 3] = 2.0        # constant column
    x[:, 7] = np.nan     # all missing
    x = np.asfortranarray(x)
    full = ik.run_pairs(x, ())
    assert (full["status"] != 0).sum() > 0
    for t in (None, 0.0):
        got = ik.run_edges(x, (), min_abs_cor=t, max_pvalue=None if t is not None else 1.0)
        assert not np.isin(got["i"], [3, 7]).any() and not np.isin(got["j"], [3, 7]).any()
        same(got, expected(full, 12, t, None if t is not None else 1.0, True), "degenerate")


def test_two_rows_nan_pvalue():
    """n = 2: the p-value is NaN; such a pair passes min_abs_cor alone and fails any max_pvalue"""
    x = np.asfortranarray(np.array([[1.0, 2.0, 3.0, 1.0], [2.0, 1.0, 4.0, 1.0]]))
    full = ik.run_pairs(x, ())
    ok = full["status"] == 0
    assert ok.any() and np.isnan(full["pvalue"][ok]).all()
    got = ik.run_edges(x, (), min_abs_cor=0.0)
    assert got["i"].size == int(ok.sum())
    same(got, expected(full, 4, 0.0, None, True), "n=2 min_abs_cor")
    got = ik.run_edges(x, (), min_abs_cor=0.0, max_pvalue=1.0)
    assert got["i"].size == 0


def test_csc_equals_dense():
    rng = np.random.default_rng(6)
    d = rng.normal(size=(3000, 80)) + rng.normal(size=(3000, 1))
    d[rng.random(d.shape) < 0.5] = 0.0
    a = sp.csc_matrix(d)
    gna = (np.nan, np.inf, 0.0)
    for t, al in ((0.2, None), (None, 1e-2), (0.0, None)):
        x = ik.run_edges(a, gna, min_abs_cor=t, max_pvalue=al)
        y = ik.run_edges(np.asfortranarray(d), gna, min_abs_cor=t, max_pvalue=al)
        same(x, y, f"csc t={t} a={al}")
        same(x, expected(ik.run_pairs(d, gna), 80, t, al, True), f"csc vs pairs t={t} a={al}")


def test_include_diag_comes_after_the_triangle():
    x = gen(1000, 40, "normal", 0.1, seed=9)
    full = check_grid(x, "global", "include_diag", ts=(None, 0.2), As=(None,), include_diag=True)
    got = ik.run_edges(x, (), min_abs_cor=0.0, include_diag=True)
    P = 40 * 39 // 2
    assert got["i"].size == P + 40 == full["raw"].size
    assert np.array_equal(got["i"][P:], np.arange(40)) and np.array_equal(got["j"][P:], np.arange(40))
    # (i, j) are the library's pair order
    for k in (0, 1, 38, 39, P - 1, P, P + 39):
        assert _lib.pair_from_index(40, k, include_diag=True) == (got["i"][k], got["j"][k])


def test_max_edges_limit_then_next_call_succeeds():
    x = gen(2000, 100, "normal", 0.0, seed=10)
    full = ik.run_pairs(x, ())
    want = expected(full, 100, 0.3, None, True)
    m = want["i"].size
    assert m > 10
    with pytest.raises(ik.IciktError) as e:
        ik.run_edges(x, (), min_abs_cor=0.3, max_edges=m - 1)
    assert e.value.code == _lib.ERR_LIMIT
    same(ik.run_edges(x, (), min_abs_cor=0.3, max_edges=m), want, "after the limit")
    same(ik.run_edges(x, (), min_abs_cor=0.3), want, "no limit")


def test_nothing_passes():
    x = gen(2000, 50, "normal", 0.1, seed=11)
    got = ik.run_edges(x, (), min_abs_cor=1.01, scale_max=False)
    for k in ("i", "j"):
        assert got[k].dtype == np.int32 and got[k].shape == (0,)
    for k in FIELDS:
        assert got[k].dtype == np.float64 and got[k].shape == (0,)


def _masked(table, t, a):
    sel = np.ones(len(table["cor"]), dtype=bool)
    with np.errstate(invalid="ignore"):
        if t is not None:
            sel &= np.abs(table["cor"]) >= t
        if a is not None:
            sel &= table["pvalue"] <= a
    return {k: np.asarray(v)[sel] for k, v in table.items()}


@pytest.mark.parametrize("diag_good", [True, False])
def test_ici_kendalltau_filtered_equals_masked(diag_good):
    x = gen(1500, 30, "mixed", 0.1, seed=12)
    names = [f"s{k}" for k in range(30)]
    for include_only in (None, ["s2", "s17"]):
        for scale_max in (True, False):
            kw = dict(colnames=names, return_matrix=False, diag_good=diag_good, scale_max=scale_max,
                      include_only=include_only)
            full = ik.ici_kendalltau(x, **kw)["cor"]
            for t, a in ((0.3, None), (None, 1e-3), (0.1, 0.05), (0.0, None)):
                got = ik.ici_kendalltau(x, min_abs_cor=t, max_pvalue=a, **kw)["cor"]
                want = _masked(full, t, a)
                w = f"ici_kendalltau diag_good={diag_good} include_only={include_only} scale_max={scale_max} t={t} a={a}"
                assert list(got["s1"]) == list(want["s1"]) and list(got["s2"]) == list(want["s2"]), w
                for k in FIELDS:
                    assert np.array_equal(np.asarray(got[k]).view(np.int64), want[k].view(np.int64)), f"{w}: {k}"


def test_large_case_against_run_pairs():
    """C = 20 000 at n = 2 000: 2 x 10^8 pairs, several default windows"""
    x = gen(2000, 20000, "normal", 0.1, seed=13)
    got = ik.run_edges(x, (), min_abs_cor=0.3)
    full = ik.run_pairs(x, ())
    same_max(got, full, "large")
    raw = full.pop("raw")
    cor = raw / full["max_taumax"]
    sel = (full["status"] == 0) & (np.abs(cor) >= 0.3)
    del full["status"]
    idx = np.nonzero(sel)[0]
    assert idx.size == got["i"].size > 0
    assert np.array_equal(got["cor"].view(np.int64), cor[idx].view(np.int64))
    assert np.array_equal(got["raw"].view(np.int64), raw[idx].view(np.int64))
    for k in ("pvalue", "taumax", "completeness"):
        assert np.array_equal(got[k].view(np.int64), full[k][idx].view(np.int64)), k
    C = 20000
    rows = np.arange(C, dtype=np.int64)
    row_start = rows * (2 * C - rows - 1) // 2
    i = np.searchsorted(row_start, idx, side="right") - 1
    assert np.array_equal(got["i"], i) and np.array_equal(got["j"], i + 1 + (idx - row_start[i]))
    assert got["timings"]["pairs_ms"] > 0 and got["timings"]["n_launches"] > 3
