"""The top-k all-pairs call (icikt_all_pairs_topk) on the GPU.  Every comparison is bit for bit against run_pairs on
the same input, with each column's candidates sorted on the host by the contract's order:

    candidates of c: d != c with status(min(c, d), max(c, d)) == 0,
    ranked by -abs(raw) (by="abs") or -raw (by="signed"), then d; the first k kept, the rest padded.

Windows of 1, 7 and 4096 pairs (ICIKT_EDGE_WINDOW) cut units, tiles and buckets mid-way and make the lists fill
over many windows."""
import numpy as np
import pytest
import scipy.sparse as sp

import icikendalltau_b200 as ik
from icikendalltau_b200 import _lib
from tests.test_gpu_parity import gen

pytestmark = pytest.mark.gpu

FIELDS = ("cor", "raw", "pvalue", "taumax", "completeness")


def pair_order(C):
    iu = np.triu_indices(C, 1)
    return iu[0].astype(np.int64), iu[1].astype(np.int64)


def topk_reference(C, k, by, scale_max, pi, pj, full, M, cols=None):
    """(C, k) lists from per-pair results (pi, pj, full) sorted on the host; cols: only these columns' rows"""
    ok = full["status"] == 0
    pi, pj = pi[ok], pj[ok]
    f = {name: full[name][ok] for name in ("raw", "pvalue", "taumax", "completeness")}
    col = np.concatenate([pi, pj])
    partner = np.concatenate([pj, pi])
    src = np.concatenate([np.arange(pi.size)] * 2)
    if cols is not None:
        keep = np.isin(col, cols)
        col, partner, src = col[keep], partner[keep], src[keep]
    raw = f["raw"][src]
    rank_key = -np.abs(raw) if by == "abs" else -raw  # -0.0 == 0.0: the tie goes to the partner
    order = np.lexsort((partner, rank_key, col))
    col, partner, src = col[order], partner[order], src[order]
    first = np.searchsorted(col, col, side="left")
    r = np.arange(col.size) - first
    sel = r < k
    col, partner, src, r = col[sel], partner[sel], src[sel], r[sel]
    out = dict(index=np.full((C, k), -1, dtype=np.int32))
    out.update((name, np.full((C, k), np.nan)) for name in FIELDS)
    out["index"][col, r] = partner
    for name in ("raw", "pvalue", "taumax", "completeness"):
        out[name][col, r] = f[name][src]
    out["cor"][col, r] = f["raw"][src] / M if scale_max else f["raw"][src]
    out["n_neighbors"] = np.bincount(col, minlength=C).astype(np.int32)
    return out


def same(got, want, what, rows=None):
    for name in ("index", "n_neighbors") + FIELDS:
        g, w = np.asarray(got[name]), np.asarray(want[name])
        if rows is not None:
            g, w = g[rows], w[rows]
        assert g.dtype == w.dtype and g.shape == w.shape, f"{what}: {name} {g.dtype}{g.shape} vs {w.dtype}{w.shape}"
        if g.dtype == np.float64:
            assert np.array_equal(g.view(np.int64), w.view(np.int64)), f"{what}: {name}"
        else:
            assert np.array_equal(g, w), f"{what}: {name}"


def same_max(got, M, what):
    assert np.array_equal(np.float64(got["max_taumax"]).view(np.int64), np.float64(M).view(np.int64)), what


def check_grid(x, persp, what, gna=(), ks=None, bys=("abs", "signed"), scales=(True, False), **kw):
    C = x.shape[1]
    full = ik.run_pairs(x, gna, perspective=persp, **kw)
    pi, pj = pair_order(C)
    for k in ks or (1, 5, C - 1, C + 3):
        for by in bys:
            for scale_max in scales:
                got = ik.run_topk(x, gna, k=k, by=by, scale_max=scale_max, perspective=persp, **kw)
                w = f"{what} {persp} k={k} by={by} scale_max={scale_max}"
                same(got, topk_reference(C, k, by, scale_max, pi, pj, full, full["max_taumax"]), w)
                same_max(got, full["max_taumax"], w)
    return full


SHAPES = [(2000, 300), (5000, 120), (20000, 64), (60000, 24)]  # the last one runs the in-place pair kernel


@pytest.mark.parametrize("n,C", SHAPES)
@pytest.mark.parametrize("kind", ["normal", "ties"])
def test_topk_equals_sorted_pairs(n, C, kind):
    x = gen(n, C, kind, 0.1, seed=n + C)
    for persp in ("global", "local"):
        check_grid(x, persp, f"{n}x{C} {kind}")
    if n == 60000:
        assert _lib.launch_shape(n)["variant"] == "inplace"


@pytest.mark.parametrize("window", [1, 7, 4096])
def test_small_windows(monkeypatch, window):
    monkeypatch.setenv("ICIKT_EDGE_WINDOW", str(window))
    n, C = (300, 30) if window == 1 else (2000, 120)
    x = gen(n, C, "mixed", 0.15, seed=window)
    check_grid(x, "global", f"window={window}", ks=(1, 5, C - 1))
    check_grid(x, "local", f"window={window}", ks=(3,), scales=(True,))


@pytest.mark.parametrize("window", [7, None])
def test_identical_columns_tie_on_the_partner(monkeypatch, window):
    """groups of identical columns: equal raws at the k boundary are decided by the partner"""
    if window:
        monkeypatch.setenv("ICIKT_EDGE_WINDOW", str(window))
    rng = np.random.default_rng(21)
    base = rng.normal(size=(400, 6))
    x = np.asfortranarray(base[:, rng.integers(0, 6, size=90)])
    x[:, 40:50] = -x[:, 40:50]  # negated copies: equal |raw|, opposite sign
    full = check_grid(x, "global", f"identical window={window}", ks=(1, 4, 17, 89))
    raw = full["raw"][full["status"] == 0]
    assert np.unique(np.abs(raw)).size < raw.size // 50  # ties everywhere


def test_degenerate_columns_are_nobodys_neighbours():
    rng = np.random.default_rng(5)
    x = rng.normal(size=(500, 14)) + rng.normal(size=(500, 1))
    x[:, 3] = 2.0        # a single value
    x[:, 7] = np.nan     # all missing
    x = np.asfortranarray(x)
    full = check_grid(x, "global", "degenerate", ks=(1, 5, 13, 20))
    got = ik.run_topk(x, (), k=20)
    assert got["n_neighbors"][3] == got["n_neighbors"][7] == 0
    assert (got["n_neighbors"][[c for c in range(14) if c not in (3, 7)]] == 11).all()
    assert not np.isin(got["index"], [3, 7]).any()
    assert (got["index"][3] == -1).all() and np.isnan(got["cor"][7]).all()
    assert np.isnan(full["raw"]).sum() > 0


@pytest.mark.parametrize("alternative,continuity", [("less", False), ("greater", True), ("two.sided", True)])
def test_alternative_and_continuity(alternative, continuity):
    x = gen(1500, 50, "mixed", 0.1, seed=31)
    check_grid(x, "global", f"{alternative} continuity={continuity}", ks=(5, 49), scales=(True,),
               alternative=alternative, continuity=continuity)


def test_csc_equals_dense():
    rng = np.random.default_rng(6)
    d = rng.normal(size=(3000, 80)) + rng.normal(size=(3000, 1))
    d[rng.random(d.shape) < 0.5] = 0.0
    a = sp.csc_matrix(d)
    gna = (np.nan, np.inf, 0.0)
    full = ik.run_pairs(d, gna)
    pi, pj = pair_order(80)
    for k, by in ((7, "abs"), (79, "signed")):
        x = ik.run_topk(a, gna, k=k, by=by)
        y = ik.run_topk(np.asfortranarray(d), gna, k=k, by=by)
        same(x, y, f"csc k={k} {by}")
        same(x, topk_reference(80, k, by, True, pi, pj, full, full["max_taumax"]), f"csc vs pairs k={k} {by}")


def test_k_max_with_more_columns():
    C = 1100
    x = gen(800, C, "normal", 0.05, seed=41)
    full = ik.run_pairs(x, ())
    pi, pj = pair_order(C)
    for by in ("abs", "signed"):
        got = ik.run_topk(x, (), k=_lib.TOPK_MAX, by=by)
        same(got, topk_reference(C, _lib.TOPK_MAX, by, True, pi, pj, full, full["max_taumax"]), f"k=1024 {by}")
    assert (got["n_neighbors"] == _lib.TOPK_MAX).all()


def test_one_column_and_two_rows():
    got = ik.run_topk(np.ones((10, 1)), (), k=3)
    assert (got["index"] == -1).all() and np.isnan(got["raw"]).all() and got["n_neighbors"][0] == 0
    assert np.isnan(got["max_taumax"])
    x = np.asfortranarray(np.array([[1.0, 2.0, 3.0, 1.0], [2.0, 1.0, 4.0, 1.0]]))
    check_grid(x, "global", "n=2", ks=(1, 3, 6))


def test_ici_kendalltau_topk_names():
    x = gen(1500, 30, "mixed", 0.1, seed=12)
    names = [f"s{k}" for k in range(30)]
    got = ik.ici_kendalltau_topk(x, 4, colnames=names)
    want = ik.run_topk(x, (np.nan, np.inf, 0.0), k=4)
    same(got, want, "ici_kendalltau_topk")
    assert got["neighbors"].shape == (30, 4)
    assert [[names[d] for d in row] for row in want["index"]] == got["neighbors"].tolist()


def test_large_case_against_pair_lists():
    """C = 20 000 at n = 2 000 with k = 16: 2 x 10^8 pairs over several default windows; the lists of 50 random
    columns come from run_pairs over their pair lists, the maximum from the edges call"""
    C, k = 20000, 16
    x = gen(2000, C, "normal", 0.1, seed=13)
    got = ik.run_topk(x, (), k=k)
    M = ik.run_edges(x, (), min_abs_cor=1.01)["max_taumax"]
    same_max(got, M, "large")
    cols = np.random.default_rng(14).choice(C, size=50, replace=False)
    other = [np.delete(np.arange(C), c) for c in cols]
    code = np.unique(np.concatenate([np.minimum(c, d) * C + np.maximum(c, d) for c, d in zip(cols, other)]))
    pi, pj = (code // C).astype(np.int32), (code % C).astype(np.int32)  # a pair of two chosen columns once
    full = ik.run_pairs(x, (), pi=pi, pj=pj)
    want = topk_reference(C, k, "abs", True, pi.astype(np.int64), pj.astype(np.int64), full, M, cols=cols)
    same(got, want, "large", rows=cols)
    assert (got["n_neighbors"] == k).all()
    assert got["timings"]["pairs_ms"] > 0 and got["timings"]["n_launches"] > 4
