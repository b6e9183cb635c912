"""Adjusted p-values on the GPU: the _padj edge calls and icikt_p_adjust.  Every comparison is bit for bit (int64 views
of the doubles).  The expected rows are run_pairs / run_cross on the same input, the NumPy restatement of R's p.adjust
(oracle/p_adjust.py) over all its p-values, and the mask

    status == 0 & (t is None | abs(cor) >= t) & (a is None | pvalue <= a) & (max_padj is NaN | padj <= max_padj).

The device keeps only the p-values <= max_padj; a max_padj of 1e-6 keeps few, NaN every one."""
import numpy as np
import pytest
import scipy.sparse as sp

import icikendalltau_b200 as ik
from icikendalltau_b200 import _lib, api
from oracle.p_adjust import METHODS, p_adjust
from tests.test_edges_gpu import SHAPES, late_maximum_matrix, pair_order
from tests.test_gpu_parity import gen

pytestmark = pytest.mark.gpu

NAN = float("nan")
MAX_PADJ = (NAN, 1e-6, 0.05, 1.0)
FILTERS = ((None, None, True), (0.3, None, True), (None, 1e-3, False))  # (min_abs_cor, max_pvalue, scale_max)
FIELDS = ("cor", "raw", "pvalue", "taumax", "completeness", "padj")


def expected(full, pi, pj, method, t, a, b, scale_max):
    raw, pv = full["raw"], full["pvalue"]
    padj = p_adjust(pv, method)
    cor = raw / full["max_taumax"] if scale_max else raw
    sel = full["status"] == 0
    with np.errstate(invalid="ignore"):
        if t is not None:
            sel &= np.abs(cor) >= t
        if a is not None:
            sel &= pv <= a
        if b == b:
            sel &= padj <= b
    out = dict(i=pi[sel], j=pj[sel], cor=cor[sel], padj=padj[sel], n_tests=int((~np.isnan(pv)).sum()))
    out.update((k, full[k][sel]) for k in ("raw", "pvalue", "taumax", "completeness"))
    return out


def same(got, want, what):
    assert got["n_tests"] == want["n_tests"], f"{what}: n_tests {got['n_tests']} vs {want['n_tests']}"
    for k in ("i", "j") + FIELDS:
        g, w = np.asarray(got[k]), np.asarray(want[k])
        assert g.shape == w.shape, f"{what}: {k} {g.shape} vs {w.shape}"
        if g.dtype == np.float64:
            assert np.array_equal(g.view(np.int64), w.view(np.int64)), f"{what}: {k}"
        else:
            assert np.array_equal(g, w.astype(g.dtype)), f"{what}: {k}"


def check_grid(x, persp, what, methods=METHODS, bounds=MAX_PADJ, filters=FILTERS, include_diag=False, devices=None):
    C = x.shape[1]
    full = ik.run_pairs(x, (), perspective=persp, include_diag=include_diag)
    pi, pj = pair_order(C, include_diag)
    for method in methods:
        for b in bounds:
            for t, a, scale_max in filters:
                got = ik.run_edges(x, (), min_abs_cor=t, max_pvalue=a, scale_max=scale_max, perspective=persp,
                                   include_diag=include_diag, p_adjust=method, max_padj=b, devices=devices)
                w = f"{what} {persp} {method} max_padj={b} t={t} a={a} scale_max={scale_max}"
                same(got, expected(full, pi, pj, method, t, a, b, scale_max), w)
                assert np.float64(got["max_taumax"]).view(np.int64) == np.float64(full["max_taumax"]).view(np.int64)
    return full


@pytest.mark.parametrize("n,C", SHAPES)
@pytest.mark.parametrize("kind", ["normal", "mixed", "ties"])
def test_padj_equals_oracle(n, C, kind):
    x = gen(n, C, kind, 0.1, seed=n + C + 1)
    for persp in ("global", "local"):
        check_grid(x, persp, f"{kind} {n}x{C}")


@pytest.mark.parametrize("window", [1, 7, 4096])
def test_small_windows(monkeypatch, window):
    monkeypatch.setenv("ICIKT_EDGE_WINDOW", str(window))
    n, C = (300, 40) if window == 1 else (1000, 90)
    x = gen(n, C, "mixed", 0.15, seed=window + 100)
    check_grid(x, "global", f"window={window}", bounds=(NAN, 0.05))
    check_grid(late_maximum_matrix(1200, 70, seed=5), "local", f"late maximum window={window}",
               methods=("BH", "holm"), bounds=(NAN, 0.05, 1e-6))


def test_alternative_other_every_p_zero():
    x = gen(800, 30, "normal", 0.1, seed=21)
    full = ik.run_pairs(x, (), alternative="other")
    assert (full["pvalue"][full["status"] == 0] == 0).all()
    pi, pj = pair_order(30, False)
    for method in METHODS:
        for b in (NAN, 0.0, 0.05):
            got = ik.run_edges(x, (), p_adjust=method, max_padj=b, alternative="other")
            same(got, expected(full, pi, pj, method, None, None, b, True), f"other {method} {b}")


def test_count_data_many_equal_pvalues():
    rng = np.random.default_rng(22)
    x = np.asfortranarray(rng.poisson(0.7, size=(40, 150)).astype(np.float64))
    check_grid(x, "global", "counts")


def test_degenerate_columns_nan_pvalues():
    x = gen(500, 40, "normal", 0.1, seed=23)
    x[:, 3] = 1.0  # a single unique value
    x[:, 7] = np.nan  # all missing
    x[:-1, 11] = np.nan  # one value
    full = check_grid(x, "global", "degenerate", bounds=(NAN, 0.05))
    assert np.isnan(full["pvalue"]).any()


@pytest.mark.parametrize("C", [1, 2])
def test_tiny_families(C):
    x = gen(300, C, "normal", 0.0, seed=24)
    if C == 1:  # no pair: no family
        got = ik.run_edges(x, (), p_adjust="BH")
        assert got["n_tests"] == 0 and len(got["i"]) == 0
    for include_diag in ((True,) if C == 1 else (False, True)):
        check_grid(x, "global", f"C={C}", filters=((None, None, True),), include_diag=include_diag)


def test_include_diag():
    x = gen(1000, 40, "normal", 0.1, seed=25)
    check_grid(x, "local", "include_diag", include_diag=True, bounds=(NAN, 0.05))


def test_csc_equals_dense():
    x = gen(1500, 60, "normal", 0.3, seed=26)
    x = np.where(np.isnan(x), 0.0, x)
    s = sp.csc_matrix(x)
    for method in ("BH", "BY", "holm"):
        d = ik.run_edges(x, (np.nan, np.inf, 0.0), p_adjust=method, max_padj=0.05)
        c = ik.run_edges(s, (np.nan, np.inf, 0.0), p_adjust=method, max_padj=0.05)
        same(c, d, f"csc {method}")
        assert len(d["i"]) > 0


def test_max_edges_as_the_plain_call():
    x = gen(2000, 100, "normal", 0.0, seed=27)
    full = ik.run_pairs(x, ())
    pi, pj = pair_order(100, False)
    want = expected(full, pi, pj, "BH", 0.3, None, 0.05, True)
    m = len(want["i"])
    assert m > 10
    with pytest.raises(_lib.IciktError) as e:
        ik.run_edges(x, (), min_abs_cor=0.3, p_adjust="BH", max_padj=0.05, max_edges=m - 1)
    assert e.value.code == _lib.ERR_LIMIT
    same(ik.run_edges(x, (), min_abs_cor=0.3, p_adjust="BH", max_padj=0.05, max_edges=m), want, "at the limit")


def test_multi_device_bit_for_bit():
    x = gen(2000, 120, "mixed", 0.1, seed=28)
    lists = [[0, 0], [0, 0, 0]]
    if _lib.load().icikt_device_count() > 1:
        lists.append(list(range(_lib.load().icikt_device_count())))
    for devices in lists:
        for method in METHODS:
            for b in (NAN, 0.05, 1e-6):
                one = ik.run_edges(x, (), p_adjust=method, max_padj=b)
                many = ik.run_edges(x, (), p_adjust=method, max_padj=b, devices=devices)
                same(many, one, f"devices={devices} {method} {b}")
                y = x[:, :50]
                one = ik.run_cross_edges(y, x[:, 50:], (), p_adjust=method, max_padj=b)
                many = ik.run_cross_edges(y, x[:, 50:], (), p_adjust=method, max_padj=b, devices=devices)
                same(many, one, f"cross devices={devices} {method} {b}")


def test_multi_device_more_devices_than_pairs():
    x = gen(500, 3, "normal", 0.0, seed=29)
    for method in METHODS:
        same(ik.run_edges(x, (), p_adjust=method, devices=[0, 0, 0, 0, 0]), ik.run_edges(x, (), p_adjust=method),
             f"5 devices, 3 pairs {method}")


@pytest.mark.parametrize("kind", ["normal", "ties"])
def test_cross_equals_oracle(kind):
    x = gen(3000, 70, kind, 0.1, seed=30)
    X, Y = x[:, :30], x[:, 30:]
    for persp in ("global", "local"):
        full = ik.run_cross(X, Y, (), perspective=persp)
        pi = np.repeat(np.arange(30, dtype=np.int32), 40)
        pj = np.tile(np.arange(40, dtype=np.int32), 30)
        for method in METHODS:
            for b in MAX_PADJ:
                for t, a, scale_max in FILTERS:
                    got = ik.run_cross_edges(X, Y, (), min_abs_cor=t, max_pvalue=a, scale_max=scale_max,
                                             perspective=persp, p_adjust=method, max_padj=b)
                    same(got, expected(full, pi, pj, method, t, a, b, scale_max),
                         f"cross {kind} {persp} {method} {b} {t} {a}")
    Xs = sp.csc_matrix(np.where(np.isnan(X), 0.0, X))
    d = ik.run_cross_edges(np.where(np.isnan(X), 0.0, X), Y, (np.nan, np.inf, 0.0), p_adjust="BY", max_padj=0.05)
    same(ik.run_cross_edges(Xs, Y, (np.nan, np.inf, 0.0), p_adjust="BY", max_padj=0.05), d, "cross csc")


def test_p_adjust_large_array():
    rng = np.random.default_rng(31)
    m = 10 ** 7
    p = np.round(rng.random(m) ** 3, 6)  # heavy ties
    p[rng.random(m) < 0.01] = np.nan
    for method in METHODS + ("fdr",):
        got = ik.p_adjust(p, method)
        assert np.array_equal(got.view(np.int64), p_adjust(p, method).view(np.int64)), method


def test_p_adjust_small_and_windowed_agree():
    for m in (0, 1, 2, 3, 1000):
        p = np.random.default_rng(m).random(m)
        p[::3] = np.nan
        for method in METHODS:
            assert np.array_equal(ik.p_adjust(p, method).view(np.int64), p_adjust(p, method).view(np.int64))
    x = gen(2000, 150, "ties", 0.1, seed=32)
    full = ik.run_pairs(x, ())
    for method in METHODS:
        e = ik.run_edges(x, (), p_adjust=method)  # no bound: every pair with a p-value is a row
        dev = ik.p_adjust(full["pvalue"], method)
        ok = full["status"] == 0
        assert np.array_equal(e["padj"].view(np.int64), dev[ok].view(np.int64)), method


@pytest.mark.parametrize("diag_good", [True, False])
@pytest.mark.parametrize("include_only", [False, True])
def test_ici_kendalltau_padj_column(diag_good, include_only):
    x = gen(1500, 30, "mixed", 0.1, seed=33)
    names = [f"s{c}" for c in range(30)]
    inc = (names[:12], names[5:]) if include_only else None
    plain = api.ici_kendalltau(x, return_matrix=False, colnames=names, diag_good=diag_good, include_only=inc)["cor"]
    fam = plain["s1"] != plain["s2"] if diag_good else np.ones(len(plain["s1"]), dtype=bool)
    for method in METHODS:
        want = np.zeros(len(plain["s1"]))
        want[fam] = p_adjust(plain["pvalue"][fam], method)
        got = api.ici_kendalltau(x, return_matrix=False, colnames=names, diag_good=diag_good, include_only=inc,
                                 p_adjust=method)["cor"]
        assert np.array_equal(got["padj"].view(np.int64), want.view(np.int64)), method
        for b, t in ((0.05, None), (0.05, 0.2), (1e-6, None)):
            sel = want <= b
            if t is not None:
                sel &= np.abs(plain["cor"]) >= t
            r = api.ici_kendalltau(x, return_matrix=False, colnames=names, diag_good=diag_good, include_only=inc,
                                   p_adjust=method, max_padj=b, min_abs_cor=t)["cor"]
            assert list(r["s1"]) == list(plain["s1"][sel]) and list(r["s2"]) == list(plain["s2"][sel]), (method, b)
            assert np.array_equal(r["padj"].view(np.int64), want[sel].view(np.int64)), (method, b, t)
            assert np.array_equal(r["pvalue"].view(np.int64), plain["pvalue"][sel].view(np.int64))


def test_ici_kendalltau_cross_padj_column():
    x = gen(1500, 40, "normal", 0.1, seed=34)
    X, Y = x[:, :15], x[:, 15:]
    kw = dict(xnames=[f"x{c}" for c in range(15)], ynames=[f"y{c}" for c in range(25)], return_matrix=False)
    plain = api.ici_kendalltau_cross(X, Y, **kw)["cor"]
    for method in ("BH", "BY", "bonferroni"):
        want = p_adjust(plain["pvalue"], method)
        got = api.ici_kendalltau_cross(X, Y, p_adjust=method, **kw)["cor"]
        assert np.array_equal(got["padj"].view(np.int64), want.view(np.int64))
        r = api.ici_kendalltau_cross(X, Y, p_adjust=method, max_padj=0.05, **kw)["cor"]
        sel = want <= 0.05
        assert np.array_equal(r["padj"].view(np.int64), want[sel].view(np.int64))
