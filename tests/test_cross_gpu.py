"""The cross calls (icikt_cross_pairs, icikt_cross_edges, icikt_cross_topk) on the GPU.  Every comparison is bit for
bit (int64 views of the doubles) against icikt_pair_list on the dense [X | Y] with pi = i and pj = Cx + j, the pairs in
x-major order: the per-pair result itself, masked on the host for the edges, and sorted on the host (|raw| or raw
descending, then partner ascending) for the top-k lists.  Windows of 1, 7 and 4096 pairs (ICIKT_EDGE_WINDOW) cut units
and rows of the cross order mid-way."""
import numpy as np
import pytest
import scipy.sparse as sp

import icikendalltau_b200 as ik
from icikendalltau_b200 import _lib
from tests.test_edges_gpu import late_maximum_matrix
from tests.test_gpu_parity import gen
from tests.test_launch_variants_gpu import censored, device_stats, grouped_col, tier2_matrix, tier_of, with_missing

pytestmark = pytest.mark.gpu

FIELDS = ("raw", "pvalue", "taumax", "completeness")


def dense(a):
    return np.asarray(a.toarray() if sp.issparse(a) else a, dtype=np.float64)


def reference(x, y, gna=(), lo=0, hi=None, **kw):
    """run_pairs on [X | Y] over pairs [lo, hi) of the cross order"""
    xd, yd = dense(x), dense(y)
    cx, cy = xd.shape[1], yd.shape[1]
    hi = cx * cy if hi is None else hi
    p = np.arange(lo, hi)
    pi, pj = (p // cy).astype(np.int32), (cx + p % cy).astype(np.int32)
    return ik.run_pairs(np.asfortranarray(np.hstack([xd, yd])), gna, pi=pi, pj=pj, **kw)


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.int64)


def same_pairs(got, want, what):
    for k in FIELDS:
        assert np.array_equal(bits(got[k]), bits(want[k])), f"{what}: {k}"
    assert np.array_equal(got["status"], want["status"]), f"{what}: status"
    assert bits(got["max_taumax"]) == bits(want["max_taumax"]), f"{what}: max_taumax"


@pytest.fixture
def window(monkeypatch):
    def set_window(w):
        if w is None:
            monkeypatch.delenv("ICIKT_EDGE_WINDOW", raising=False)
        else:
            monkeypatch.setenv("ICIKT_EDGE_WINDOW", str(w))
    yield set_window


def degenerate_pair(seed, n=400, cx=5, cy=6):
    """X and Y from one signal, with an all-missing and a single-value column on each side and an X column repeated
    in Y"""
    x = gen(n, cx + cy, "mixed", 0.1, seed)
    x, y = x[:, :cx].copy(), x[:, cx:].copy()
    x[:, 1] = np.nan
    y[:, 4] = np.nan
    x[:, 3] = 2.5
    y[:, 0] = np.where(np.isnan(y[:, 0]), np.nan, -1.0)
    y[:, 2] = x[:, 0]
    return np.asfortranarray(x), np.asfortranarray(y)


# ---------------------------------------------------------------- icikt_cross_pairs
@pytest.mark.parametrize("w", [1, 7, 4096])
@pytest.mark.parametrize("persp", ["global", "local"])
def test_pairs_equal_pair_list(window, persp, w):
    window(w)
    x, y = degenerate_pair(seed=w)
    for alt, cont in (("two.sided", False), ("less", True), ("greater", False)):
        kw = dict(perspective=persp, alternative=alt, continuity=cont)
        got = ik.run_cross(x, y, (np.nan,), **kw)
        want = reference(x, y, (np.nan,), **kw)
        same_pairs(got, want, f"{persp} {alt} continuity={cont} window={w}")
        assert (got["status"] != 0).sum() > 0


@pytest.mark.parametrize("lo,hi", [(0, 1), (3, 4), (5, 29), (29, 30), (6, 12), (0, 30), (17, 17)])
def test_pair_slices(window, lo, hi):
    window(7)
    x, y = degenerate_pair(seed=5)
    got = ik.run_cross(x, y, (), pair_lo=lo, pair_hi=hi)
    assert got["raw"].size == hi - lo
    if hi > lo:
        same_pairs(got, reference(x, y, (), lo, hi), f"[{lo}, {hi})")
    else:
        assert np.isnan(got["max_taumax"])


@pytest.mark.parametrize("cx,cy", [(1, 9), (9, 1), (1, 1)])
def test_one_column_sides(window, cx, cy):
    for w in (1, 4096):
        window(w)
        m = gen(300, cx + cy, "ties", 0.05, cx * 10 + cy)
        x, y = m[:, :cx], m[:, cx:]
        for persp in ("global", "local"):
            same_pairs(ik.run_cross(x, y, (), perspective=persp), reference(x, y, (), perspective=persp),
                       f"{cx} x {cy} {persp} window={w}")


def test_csc_sides_against_dense(window):
    rng = np.random.default_rng(8)
    a = sp.random(500, 7, density=0.3, format="csc", random_state=1)
    b = sp.random(500, 9, density=0.5, format="csc", random_state=2)
    a.data = np.round(a.data * 5)
    gna = (np.nan, np.inf, 0.0)
    for w in (7, 4096):
        window(w)
        for x, y in ((a, dense(b)), (dense(a), b), (a, b)):
            want = reference(x, y, gna)
            same_pairs(ik.run_cross(x, y, gna), want, f"sparse x={sp.issparse(x)} y={sp.issparse(y)} window={w}")
    # an all-stored-zero column and one with nothing stored
    c = sp.csc_matrix(np.column_stack([np.zeros(500), rng.normal(size=500)]))
    same_pairs(ik.run_cross(c, a, gna), reference(c, a, gna), "empty CSC columns")


TIERS = {
    "tier 0": lambda: censored(3000, [0, 5, 900, 2999, 1500, 40], seed=2),
    "tier 1 in place": lambda: np.asfortranarray(np.column_stack([
        grouped_col(np.random.default_rng(1), 60000, 10, 400, n_na=5000), np.random.default_rng(2).standard_normal(60000),
        with_missing(np.random.default_rng(3), np.random.default_rng(4).standard_normal(60000), 3000)])),
    "tier 2": lambda: tier2_matrix(4096, 17, 200, seed=3)[1],
}


@pytest.mark.parametrize("case,tier", [("tier 0", 0), ("tier 1 in place", 1), ("tier 2", 2)])
def test_tiers(window, case, tier):
    m = TIERS[case]()
    assert tier_of(device_stats(m), m.shape[0]) == tier, case
    cx = m.shape[1] // 2
    x, y = np.asfortranarray(m[:, :cx]), np.asfortranarray(m[:, cx:])
    for w in (7, None):
        window(w)
        for persp in ("global", "local"):
            same_pairs(ik.run_cross(x, y, (), perspective=persp), reference(x, y, (), perspective=persp),
                       f"{case} {persp} window={w}")


# ---------------------------------------------------------------- icikt_cross_edges
def masked(full, cx, cy, t, a, scale_max):
    raw, pv = full["raw"], full["pvalue"]
    cor = raw / full["max_taumax"] if scale_max else raw
    sel = full["status"] == 0
    with np.errstate(invalid="ignore"):
        if t is not None:
            sel &= np.abs(cor) >= t
        if a is not None:
            sel &= pv <= a
    p = np.nonzero(sel)[0]
    out = dict(i=(p // cy).astype(np.int32), j=(p % cy).astype(np.int32), cor=cor[sel])
    out.update((k, full[k][sel]) for k in FIELDS)
    return out


def same_edges(got, want, what):
    for k in ("i", "j"):
        assert np.array_equal(got[k], want[k]), f"{what}: {k}"
    for k in ("cor",) + FIELDS:
        assert np.array_equal(bits(got[k]), bits(want[k])), f"{what}: {k}"


@pytest.mark.parametrize("w", [1, 7, 4096])
def test_edges_equal_masked_pairs(window, w):
    window(w)
    x, y = degenerate_pair(seed=11, cx=7, cy=9)
    cx, cy = x.shape[1], y.shape[1]
    for persp in ("global", "local"):
        full = reference(x, y, (), perspective=persp)
        for scale_max in (True, False):
            for t, a in ((None, None), (0.3, None), (None, 1e-2), (0.5, 1e-3), (1.01, None)):
                got = _lib.run_cross_edges(x, y, (), t, a, scale_max, perspective=persp)
                what = f"{persp} window={w} scale_max={scale_max} t={t} a={a}"
                same_edges(got, masked(full, cx, cy, t, a, scale_max), what)
                assert bits(got["max_taumax"]) == bits(full["max_taumax"]), what


@pytest.mark.parametrize("w", [1, 7, 4096])
def test_edges_late_maximum_and_limit(window, w):
    window(w)
    # every column but the last of each side has missing rows: the pair of largest taumax comes last in cross order
    m = late_maximum_matrix(800, 24, seed=3)
    x, y = np.asfortranarray(np.column_stack([m[:, :11], m[:, 22]])), np.asfortranarray(np.column_stack([m[:, 11:22], m[:, 23]]))
    cx, cy = x.shape[1], y.shape[1]
    full = reference(x, y, ())
    tm = full["taumax"]
    assert np.nanargmax(tm) == tm.size - 1 and tm[-1] == 1.0
    t = float(np.quantile(np.abs(full["raw"][full["status"] == 0]), 0.8))
    early = (full["status"] == 0) & (np.abs(full["raw"]) >= t * np.nanmax(tm[:-1])) & (np.abs(full["raw"]) < t)
    assert early.sum() > 0  # rows the running maximum keeps and the final one removes
    want = masked(full, cx, cy, t, None, True)
    same_edges(_lib.run_cross_edges(x, y, (), t, None, True), want, f"late maximum window={w}")
    m_pass = want["i"].size
    assert m_pass > 1
    if w == 4096:  # one window: the rows held are the final ones (smaller windows may hold more, as documented)
        same_edges(_lib.run_cross_edges(x, y, (), t, None, True, max_edges=m_pass), want, "max_edges = count")
        with pytest.raises(ik.IciktError) as e:
            _lib.run_cross_edges(x, y, (), t, None, True, max_edges=m_pass - 1)
        assert e.value.code == _lib.ERR_LIMIT
    want = masked(full, cx, cy, None, 1e-2, True)
    with pytest.raises(ik.IciktError) as e:  # without a cor bound the held count is exact in every window
        _lib.run_cross_edges(x, y, (), None, 1e-2, True, max_edges=want["i"].size - 1)
    assert e.value.code == _lib.ERR_LIMIT
    same_edges(_lib.run_cross_edges(x, y, (), None, 1e-2, True, max_edges=want["i"].size), want, "after the limit")


# ---------------------------------------------------------------- icikt_cross_topk
def host_lists(full, cx, cy, k, by, scale_max, side):
    """the lists of one side by a host lexsort of the per-pair cross result"""
    raw = full["raw"].reshape(cx, cy)
    ok = (full["status"] == 0).reshape(cx, cy)
    vals = {f: full[f].reshape(cx, cy) for f in FIELDS}
    if side == "y":
        raw, ok = raw.T, ok.T
        vals = {f: v.T for f, v in vals.items()}
    C = raw.shape[0]
    out = dict(index=np.full((C, k), -1, dtype=np.int32), n_neighbors=np.zeros(C, dtype=np.int32))
    out.update((f, np.full((C, k), np.nan)) for f in ("cor",) + FIELDS)
    for c in range(C):
        d = np.nonzero(ok[c])[0]
        r = raw[c, d]
        o = d[np.lexsort((d, -np.abs(r) if by == "abs" else -(r + 0.0)))][:k]
        h = o.size
        out["index"][c, :h] = o
        out["n_neighbors"][c] = h
        for f in FIELDS:
            out[f][c, :h] = vals[f][c, o]
        out["cor"][c, :h] = vals["raw"][c, o] / full["max_taumax"] if scale_max else vals["raw"][c, o]
    return out


def same_lists(got, want, what):
    assert np.array_equal(got["index"], want["index"]), f"{what}: index"
    assert np.array_equal(got["n_neighbors"], want["n_neighbors"]), f"{what}: n_neighbors"
    for f in ("cor",) + FIELDS:
        assert np.array_equal(bits(got[f]), bits(want[f])), f"{what}: {f}"


@pytest.mark.parametrize("w", [1, 7, 4096])
@pytest.mark.parametrize("by", ["abs", "signed"])
def test_topk_equal_host_lexsort(window, w, by):
    window(w)
    x, y = degenerate_pair(seed=21, cx=6, cy=9)
    x[:, 5] = np.round(x[:, 5])  # equal raws with different partners
    y[:, 6] = np.round(y[:, 6])
    cx, cy = x.shape[1], y.shape[1]
    full = reference(x, y, ())
    for k in (1, 4, 12):  # 12 > both widths: padding
        for side in ("x", "y", "both"):
            got = _lib.run_cross_topk(x, y, (), k, by, True, side)
            assert set(got) - {"max_taumax", "timings"} == {"x": {"x_side"}, "y": {"y_side"},
                                                            "both": {"x_side", "y_side"}}[side]
            assert bits(got["max_taumax"]) == bits(full["max_taumax"])
            for s in ("x", "y"):
                if s + "_side" in got:
                    same_lists(got[s + "_side"], host_lists(full, cx, cy, k, by, True, s),
                               f"by={by} window={w} k={k} side={side}: {s} side")


def test_topk_k_1024_wide_reference(window):
    window(None)
    m = gen(200, 3 + 1100, "ties", 0.05, 31)
    x, y = m[:, :3], m[:, 3:]
    full = reference(x, y, ())
    got = _lib.run_cross_topk(x, y, (), 1024, "abs", False, "both")
    same_lists(got["x_side"], host_lists(full, 3, 1100, 1024, "abs", False, "x"), "k=1024 x side")
    same_lists(got["y_side"], host_lists(full, 3, 1100, 1024, "abs", False, "y"), "k=1024 y side (padded)")
    window(7)
    got = _lib.run_cross_topk(x, y, (), 1024, "signed", True, "x")
    same_lists(got["x_side"], host_lists(full, 3, 1100, 1024, "signed", True, "x"), "k=1024 window=7")


# ---------------------------------------------------------------- Python layer on the device
def test_api_full_and_long_table():
    x, y = degenerate_pair(seed=41)
    xn, yn = [f"q{c}" for c in range(x.shape[1])], [f"r{c}" for c in range(y.shape[1])]
    with pytest.warns(RuntimeWarning):
        got = ik.ici_kendalltau_cross(x, y, xnames=xn, ynames=yn)
    full = reference(x, y, (np.nan, np.inf, 0.0))
    for f in FIELDS:
        assert np.array_equal(bits(got[f]).ravel(), bits(full[f]))
        assert got[f].shape == (x.shape[1], y.shape[1])
    assert np.array_equal(bits(got["cor"]).ravel(), bits(full["raw"] / full["max_taumax"]))
    tab = ik.ici_kendalltau_cross(x, y, xnames=xn, ynames=yn, return_matrix=False, min_abs_cor=0.4)["cor"]
    sel = (full["status"] == 0) & (np.abs(full["raw"] / full["max_taumax"]) >= 0.4)
    p = np.nonzero(sel)[0]
    assert list(tab["s1"]) == [xn[i] for i in p // y.shape[1]] and list(tab["s2"]) == [yn[j] for j in p % y.shape[1]]
    top = ik.ici_kendalltau_cross_topk(x, y, 3, side="both", xnames=xn, ynames=yn)
    assert top["x"]["neighbors"][0, 0] in yn and top["y"]["neighbors"][0, 0] in xn
