"""The component calls on the GPU.  For every filter, the labels and n_components are compared as integers against
scipy's connected components of the graph of run_pairs / run_cross masked on the host with the count predicate
(labels canonicalised to the smallest vertex); n_pass and the degrees must equal the count call's.  Windows of 1, 7
and 4096 pairs, a bridging pair that is the last of the order, all-pass, none-pass and planted groups, cross calls
with either label table NULL, and the _multi twins, which must return the one-device arrays exactly."""
import ctypes

import numpy as np
import pytest
import scipy.sparse as sp
from scipy.sparse.csgraph import connected_components

import icikendalltau_b200 as ik
from icikendalltau_b200 import _lib
from tests.test_edge_counts_gpu import degenerate_matrix, filters_of, mask, pair_order
from tests.test_gpu_parity import gen

pytestmark = [pytest.mark.gpu, pytest.mark.filterwarnings("ignore::RuntimeWarning")]

GNA = (np.nan, np.inf, 0.0)


@pytest.fixture
def window(monkeypatch):
    def set_window(w):
        if w is None:
            monkeypatch.delenv("ICIKT_EDGE_WINDOW", raising=False)
        else:
            monkeypatch.setenv("ICIKT_EDGE_WINDOW", str(w))
    return set_window


def reference(V, a, b):
    """(labels as the smallest vertex of each component, number of components)"""
    g = sp.coo_matrix((np.ones(len(a)), (a, b)), shape=(V, V))
    n, lab = connected_components(g, directed=False)
    first = np.full(n, V, dtype=np.int64)
    np.minimum.at(first, lab, np.arange(V))
    return first[lab].astype(np.int32), n


def planted(n, C, groups, seed):
    """C columns in `groups` blocks, each block a shared signal plus noise: strong pairs within a block only"""
    rng = np.random.default_rng(seed)
    g = rng.integers(0, groups, C)
    base = rng.normal(size=(n, groups))
    return np.asfortranarray(base[:, g] + 0.5 * rng.normal(size=(n, C)))


def check_all_pairs(x, full, gna=(), persp="global", include_diag=False, filters=None, devices=None):
    C = x.shape[1]
    filters = filters or filters_of(full)
    got = ik.run_count_edges(x, gna, filters, devices=devices, perspective=persp, include_diag=include_diag,
                             want_components=True)
    cnt = ik.run_count_edges(x, gna, filters, devices=devices, perspective=persp, include_diag=include_diag)
    for k in ("n_pass", "degree", "status_counts"):
        assert np.array_equal(got[k], cnt[k]), k
    assert got["component"].shape == (C, len(filters)) and got["component"].dtype == np.int32
    pi, pj = pair_order(C, include_diag)
    for f, (t, a) in enumerate(filters):
        sel = mask(full, t, a)
        lab, n = reference(C, pi[sel], pj[sel])
        assert np.array_equal(got["component"][:, f], lab), (f, t, a)
        assert got["n_components"][f] == n, (f, t, a)
    return got


@pytest.mark.parametrize("persp", ["global", "local"])
@pytest.mark.parametrize("include_diag", [False, True])
def test_dense_against_pairs(persp, include_diag):
    x = degenerate_matrix(1500, 70, seed=11)
    full = ik.run_pairs(x, (), perspective=persp, include_diag=include_diag)
    got = check_all_pairs(x, full, (), persp, include_diag)
    assert (got["component"][1] == 1).all() and (got["component"][3] == 3).all()  # degenerate: alone


@pytest.mark.parametrize("include_diag", [False, True])
def test_csc_against_dense(include_diag):
    x = gen(2000, 90, "mixed", 0.05, seed=8)
    x[np.random.default_rng(8).random(x.shape) < 0.4] = 0.0
    x[:, 7] = 0.0
    full = ik.run_pairs(x, GNA, include_diag=include_diag)
    got = check_all_pairs(sp.csc_matrix(x), full, GNA, include_diag=include_diag)
    dense = ik.run_count_edges(x, GNA, filters_of(full), include_diag=include_diag, want_components=True)
    assert np.array_equal(got["component"], dense["component"])
    assert np.array_equal(got["n_components"], dense["n_components"])


def test_zero_raws_on_the_threshold():
    x = np.asfortranarray(np.random.default_rng(5).integers(0, 4, size=(6, 60)).astype(np.float64))
    full = ik.run_pairs(x, (), include_diag=True)
    check_all_pairs(x, full, (), include_diag=True)


@pytest.mark.parametrize("w", [1, 7, 4096])
def test_small_windows(window, w):
    window(w)
    n, C = (300, 30) if w == 1 else (1200, 110)
    x = degenerate_matrix(n, C, seed=w, kind="mixed")
    for persp, diag in (("global", w == 7), ("local", False)):
        check_all_pairs(x, ik.run_pairs(x, (), perspective=persp, include_diag=diag), (), persp, diag)


@pytest.mark.parametrize("w", [7, 4096, None])
def test_bridge_is_the_last_pair(window, w):
    """a chain into a planted group whose last link is the last pair of the order: the even columns below 40 are
    noisy copies of a signal s, column 118 is s plus more noise and column 119 is 118 plus noise.  At |raw| >= 0.54,
    118 passes with every even column (tau about 0.6), 119 with 118 (about 0.65) and with nothing else (about 0.48 with
    the group); the odd columns below 40 are a second group and the rest independent.  Column 119 reaches the group
    through pair (118, 119) only, the last pair of the order, so a lost union of the last tile shows as its own
    component."""
    window(w)
    n = 2000
    rng = np.random.default_rng(2)
    x = rng.normal(size=(n, 120))
    sig = rng.normal(size=n)
    x[:, 0:40:2] = sig[:, None] + 1e-2 * rng.normal(size=(n, 20))
    x[:, 3:40:2] = x[:, [1]] + 1e-2 * rng.normal(size=(n, 19))
    x[:, 118] = sig + np.sqrt(0.5) * rng.normal(size=n)
    x[:, 119] = x[:, 118] + np.sqrt(0.5) * rng.normal(size=n)
    x = np.asfortranarray(x)
    full = ik.run_pairs(x, ())
    filters = [(0.54, None), (0.54, 1e-6), (0.7, None)]
    pi, pj = pair_order(120, False)
    at_119 = (pi == 119) | (pj == 119)
    for t, a in filters[:2]:  # the construction: 119's one edge is the last pair
        sel = mask(full, t, a)
        assert np.flatnonzero(sel & at_119).tolist() == [pi.size - 1], (t, a)
        assert (sel & (pj == 118) & (pi < 40)).sum() == 20, (t, a)  # 118 with every even column below 40
    assert not (mask(full, 0.7, None) & ((pi == 118) | at_119)).any()
    got = check_all_pairs(x, full, (), filters=filters)
    for f in (0, 1):
        assert got["n_components"][f] == 2 + 78 and got["component"][119, f] == 0 and got["component"][118, f] == 0
        assert (got["component"][1:40:2, f] == 1).all()
    assert got["n_components"][2] == 2 + 80 and got["component"][119, 2] == 119


def test_all_pass_none_pass_and_planted_groups():
    x = planted(1000, 150, 5, seed=4)
    full = ik.run_pairs(x, ())
    filters = [(None, None), (0.0, None), (1.01, None), (None, -1.0)] + \
              [(float(t), None) for t in np.linspace(0.05, 0.6, 30)]
    got = check_all_pairs(x, full, (), filters=filters)
    assert (got["n_components"][:2] == 1).all() and not got["component"][:, :2].any()
    assert (got["n_components"][2:4] == 150).all()
    assert np.array_equal(got["component"][:, 2], np.arange(150))
    assert (got["n_components"] >= 5).sum() > 5  # the groups survive part of the grid


def test_one_column():
    x = gen(100, 1, "normal", 0.0, seed=1)
    for diag in (False, True):
        got = ik.run_count_edges(x, (), [(None, None)], include_diag=diag, want_components=True)
        assert got["component"][0, 0] == 0 and got["n_components"][0] == 1


# ---------------------------------------------------------------- cross calls

def check_cross(x, y, gna=(), persp="global", filters=None, devices=None):
    cx, cy = x.shape[1], y.shape[1]
    full = ik.run_cross(x, y, gna, perspective=persp)
    filters = filters or filters_of(full)
    got = ik.run_cross_count_edges(x, y, gna, filters, devices=devices, perspective=persp, want_components=True)
    cnt = ik.run_cross_count_edges(x, y, gna, filters, devices=devices, perspective=persp)
    for k in ("n_pass", "x_degree", "y_degree", "status_counts"):
        assert np.array_equal(got[k], cnt[k]), k
    pi, pj = np.repeat(np.arange(cx), cy), np.tile(np.arange(cy), cx) + cx
    for f, (t, a) in enumerate(filters):
        sel = mask(full, t, a)
        lab, n = reference(cx + cy, pi[sel], pj[sel])
        assert np.array_equal(got["x_component"][:, f], lab[:cx]), (f, t, a)
        assert np.array_equal(got["y_component"][:, f], lab[cx:]), (f, t, a)
        assert got["n_components"][f] == n, (f, t, a)
    return got


@pytest.mark.parametrize("persp", ["global", "local"])
@pytest.mark.parametrize("w", [1, 7, 4096, None])
def test_cross_against_pairs(window, persp, w):
    window(w)
    n = 300 if w == 1 else 1200
    xy = degenerate_matrix(n, 50 if w == 1 else 130, seed=21)
    x, y = xy[:, :20 if w == 1 else 55], xy[:, 20 if w == 1 else 55:]
    check_cross(x, y, (), persp)


def test_cross_csc_and_one_side_null():
    x = gen(1500, 40, "mixed", 0.05, seed=9)
    x[np.random.default_rng(9).random(x.shape) < 0.3] = 0.0
    y = planted(1500, 33, 3, seed=10)
    got = check_cross(sp.csc_matrix(x), y, GNA)
    L = _lib.load()
    full = ik.run_cross(x, y, GNA)
    f = filters_of(full)
    arr, T = _lib._count_filters(f)
    xi, yi, n, cx, cy, keep = _lib._cross_inputs(x, y)
    o = _lib.make_opts()
    for side in (0, 1):
        tab = np.zeros(((cx, cy)[side], T), dtype=np.int32)
        ncomp = np.zeros(T, dtype=np.int64)
        npass = np.zeros(T, dtype=np.int64)
        labels = [tab.ctypes.data, None] if side == 0 else [None, tab.ctypes.data]
        g, gp, ng = _lib._global_na_array(GNA)
        assert L.icikt_cross_components(ctypes.byref(xi), ctypes.byref(yi), n, gp, ng, ctypes.byref(o),
                                        arr, T, npass.ctypes.data, None, None, *labels, ncomp.ctypes.data, None,
                                        None, None) == 0
        assert np.array_equal(tab, got["x_component" if side == 0 else "y_component"])
        assert np.array_equal(ncomp, got["n_components"]) and np.array_equal(npass, got["n_pass"])


# ---------------------------------------------------------------- several devices

@pytest.mark.parametrize("w", [7, None])
def test_multi_equals_one_device(window, w):
    window(w)
    x = planted(1500, 100, 4, seed=31)
    x[:, 5] = np.nan
    for diag in (False, True):
        f = filters_of(ik.run_pairs(x, (), include_diag=diag))
        one = ik.run_count_edges(x, (), f, include_diag=diag, want_components=True)
        for devs in ([0, 0], [0, 0, 0]):
            got = ik.run_count_edges(x, (), f, devices=devs, include_diag=diag, want_components=True)
            for k in ("n_pass", "degree", "component", "n_components"):
                assert np.array_equal(got[k], one[k]), (devs, k)
    x, y = x[:, :45], x[:, 45:]
    f = filters_of(ik.run_cross(x, y))
    one = ik.run_cross_count_edges(x, y, (), f, want_components=True)
    for devs in ([0, 0], [0, 0, 0]):
        got = ik.run_cross_count_edges(x, y, (), f, devices=devs, want_components=True)
        for k in ("n_pass", "x_component", "y_component", "n_components"):
            assert np.array_equal(got[k], one[k]), (devs, k)


# ---------------------------------------------------------------- public API

TS, PS = [0.05, 0.2, 0.6], [None, 1e-3, 0.5]


@pytest.mark.parametrize("diag_good", [True, False])
def test_api_matches_long_table(diag_good):
    x = planted(900, 40, 4, seed=41)
    x[:, 2] = np.nan
    names = [f"S{i}" for i in range(40)]
    got = ik.ici_kendalltau_edge_counts(x, min_abs_cor=TS, max_pvalue=PS, diag_good=diag_good, colnames=names,
                                        components=True)
    assert got["component"].shape == (40, 3, 3) and got["n_components"].shape == (3, 3)
    index = {s: k for k, s in enumerate(names)}
    for u, t in enumerate(TS):
        for v, p in enumerate(PS):
            tab = ik.ici_kendalltau(x, return_matrix=False, scale_max=False, min_abs_cor=t, max_pvalue=p,
                                    diag_good=diag_good, colnames=names)["cor"]
            s1 = np.array([index[s] for s in tab["s1"]], dtype=np.int64)
            s2 = np.array([index[s] for s in tab["s2"]], dtype=np.int64)
            lab, n = reference(40, s1, s2)
            assert np.array_equal(got["component"][:, u, v], lab), (t, p)
            assert got["n_components"][u, v] == n and got["largest_component"][u, v] == np.bincount(lab).max()
    plain = ik.ici_kendalltau_edge_counts(x, min_abs_cor=TS, max_pvalue=PS, diag_good=diag_good, colnames=names)
    assert "component" not in plain and np.array_equal(plain["degree"], got["degree"])


def test_cross_api_matches_long_table():
    xy = planted(900, 50, 3, seed=43)
    x, y = xy[:, :22], xy[:, 22:]
    xn, yn = [f"X{i}" for i in range(22)], [f"Y{i}" for i in range(28)]
    got = ik.ici_kendalltau_cross_edge_counts(x, y, min_abs_cor=TS, max_pvalue=PS, xnames=xn, ynames=yn,
                                              components=True)
    index = {s: k for k, s in enumerate(xn + yn)}
    for u, t in enumerate(TS):
        for v, p in enumerate(PS):
            tab = ik.ici_kendalltau_cross(x, y, return_matrix=False, scale_max=False, min_abs_cor=t, max_pvalue=p,
                                          xnames=xn, ynames=yn)["cor"]
            s1 = np.array([index[s] for s in tab["s1"]], dtype=np.int64)
            s2 = np.array([index[s] for s in tab["s2"]], dtype=np.int64)
            lab, n = reference(50, s1, s2)
            assert np.array_equal(got["x_component"][:, u, v], lab[:22]), (t, p)
            assert np.array_equal(got["y_component"][:, u, v], lab[22:]), (t, p)
            assert got["n_components"][u, v] == n and got["largest_component"][u, v] == np.bincount(lab).max()
