"""The edge-count calls on the GPU.  Every count is compared as an integer, with no tolerance, against two references
on the same input:

  * the per-pair call (run_pairs / run_cross), masked on the host with the predicate of the filtered call without
    scale_max: status == 0 & (t is None | abs(raw) >= t) & (a is None | pvalue <= a);
  * the filtered call itself (run_edges / run_cross_edges, scale_max=False) with each filter alone: its row count and
    the bincounts of its endpoints (a diagonal row counted once).

Windows of 1, 7 and 4096 pairs (ICIKT_EDGE_WINDOW) cut units and tiles mid-way; one matrix has every passing pair in
the last window.  The _multi twins must return the one-device arrays exactly."""
import numpy as np
import pytest
import scipy.sparse as sp

import icikendalltau_b200 as ik
from icikendalltau_b200 import _lib
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


def pair_order(C, include_diag):
    iu = np.triu_indices(C, 1)
    pi, pj = iu[0].astype(np.int64), iu[1].astype(np.int64)
    if include_diag:
        d = np.arange(C, dtype=np.int64)
        pi, pj = np.concatenate([pi, d]), np.concatenate([pj, d])
    return pi, pj


def mask(full, t, a):
    sel = full["status"] == 0
    with np.errstate(invalid="ignore"):
        if t is not None:
            sel &= np.abs(full["raw"]) >= t
        if a is not None:
            sel &= full["pvalue"] <= a
    return sel


def filters_of(full):
    """bounds on the data's own values: thresholds equal to exact |raw| and p-values of some pairs, zero of both
    signs, one bound, the other or none"""
    ok = full["status"] == 0
    raws = np.abs(full["raw"][ok])
    pvs = full["pvalue"][ok]
    ts = [None, 0.0, -0.0, 0.2, 1.0]
    As = [None, 0.0, -0.0, 0.05]
    if raws.size:
        ts += [float(v) for v in np.quantile(raws, [0.5, 0.9], method="nearest")]
        As += [float(v) for v in np.quantile(pvs, [0.1, 0.5], method="nearest")]
    return [(t, a) for t in ts for a in As][:64]


def bits(v):
    return np.float64(v).view(np.int64)


def check_all_pairs(x, full, gna=(), persp="global", include_diag=False, filters=None, devices=None, vs_edges=True):
    C = x.shape[1]
    filters = filters or filters_of(full)
    got = ik.run_count_edges(x, gna, filters, devices=devices, perspective=persp, include_diag=include_diag)
    pi, pj = pair_order(C, include_diag)
    assert got["n_pass"].shape == (len(filters),) and got["degree"].shape == (C, len(filters))
    for f, (t, a) in enumerate(filters):
        sel = mask(full, t, a)
        deg = np.bincount(pi[sel], minlength=C) + np.bincount(pj[sel & (pi != pj)], minlength=C)
        assert got["n_pass"][f] == int(sel.sum()), (f, t, a)
        assert np.array_equal(got["degree"][:, f], deg), (f, t, a)
        if vs_edges and f % 7 == 0:  # the filtered call walks the pairs once per filter: a sample of them
            e = ik.run_edges(x, gna, min_abs_cor=t, max_pvalue=a, scale_max=False, perspective=persp,
                             include_diag=include_diag)
            ei, ej = e["i"].astype(np.int64), e["j"].astype(np.int64)
            assert got["n_pass"][f] == ei.size, (f, t, a)
            assert np.array_equal(got["degree"][:, f],
                                  np.bincount(ei, minlength=C) + np.bincount(ej[ei != ej], minlength=C)), (f, t, a)
    assert np.array_equal(got["status_counts"], np.bincount(full["status"], minlength=_lib.NSTATUS)[:_lib.NSTATUS])
    assert bits(got["max_taumax"]) == bits(full["max_taumax"])
    return got


def degenerate_matrix(n, C, seed, kind="ties"):
    """ties, an all-missing column and a single-valued one"""
    x = gen(n, C, kind, 0.1, seed)
    x[:, 1] = np.nan
    x[:, 3] = 2.0
    return np.asfortranarray(x)


@pytest.mark.parametrize("persp", ["global", "local"])
@pytest.mark.parametrize("include_diag", [False, True])
def test_dense_against_pairs_and_edges(persp, include_diag):
    x = degenerate_matrix(1500, 70, seed=11)
    full = ik.run_pairs(x, (), perspective=persp, include_diag=include_diag)
    assert (full["status"] == 1).any() and (full["status"] == 3).any()
    check_all_pairs(x, full, (), persp, include_diag)


def test_zero_raws_on_the_threshold():
    """short integer columns: many pairs have raw == 0 exactly, counted by thresholds 0.0 and -0.0"""
    x = np.asfortranarray(np.random.default_rng(5).integers(0, 4, size=(6, 60)).astype(np.float64))
    full = ik.run_pairs(x, (), include_diag=True)
    assert ((full["raw"] == 0) & (full["status"] == 0)).any()
    check_all_pairs(x, full, (), include_diag=True)


@pytest.mark.parametrize("include_diag", [False, True])
def test_csc_against_dense(include_diag):
    x = gen(2000, 90, "mixed", 0.05, seed=8)
    x[np.random.default_rng(8).random(x.shape) < 0.4] = 0.0
    x[:, 7] = 0.0  # no stored entry: every value missing under GNA
    full = ik.run_pairs(x, GNA, include_diag=include_diag)
    got = check_all_pairs(sp.csc_matrix(x), full, GNA, include_diag=include_diag, vs_edges=False)
    dense = ik.run_count_edges(x, GNA, filters_of(full), include_diag=include_diag)
    for k in ("n_pass", "degree", "status_counts"):
        assert np.array_equal(got[k], dense[k]), k


@pytest.mark.parametrize("w", [1, 7, 4096])
def test_small_windows(window, w):
    window(w)
    n, C = (300, 30) if w == 1 else (1200, 110)
    x = degenerate_matrix(n, C, seed=w, kind="mixed")
    for persp, diag in (("global", w == 7), ("local", False)):
        full = ik.run_pairs(x, (), perspective=persp, include_diag=diag)
        check_all_pairs(x, full, (), persp, diag)


@pytest.mark.parametrize("w", [7, 4096, None])
def test_every_passing_pair_in_the_last_window(window, w):
    """independent columns but the last two, which are equal: the one pair with |raw| = 1 is the last of the order"""
    window(w)
    rng = np.random.default_rng(2)
    x = rng.normal(size=(800, 120))
    x[:, -1] = x[:, -2]
    x = np.asfortranarray(x)
    full = ik.run_pairs(x, ())
    filters = [(0.99, None), (1.0, 1e-30), (0.99, 0.0)]
    got = check_all_pairs(x, full, (), filters=filters)
    assert got["n_pass"][0] == 1 and got["degree"][-1, 0] == 1 and got["degree"][:-2].sum() == 0


def test_64_filters_and_null_degree():
    x = gen(1000, 80, "normal", 0.0, seed=4)
    full = ik.run_pairs(x, ())
    filters = [(float(t), None) for t in np.linspace(0.0, 0.63, 64)]
    got = check_all_pairs(x, full, (), filters=filters, vs_edges=False)
    bare = ik.run_count_edges(x, (), filters, want_degree=False)
    assert bare["degree"] is None and np.array_equal(bare["n_pass"], got["n_pass"])
    assert np.array_equal(bare["status_counts"], got["status_counts"])


def test_one_column():
    x = gen(100, 1, "normal", 0.0, seed=1)
    got = ik.run_count_edges(x, (), [(None, None)])
    assert got["n_pass"][0] == 0 and got["degree"].sum() == 0 and np.isnan(got["max_taumax"])
    got = ik.run_count_edges(x, (), [(None, None)], include_diag=True)
    full = ik.run_pairs(x, (), include_diag=True)
    assert got["n_pass"][0] == int((full["status"] == 0).sum())


# ---------------------------------------------------------------- cross calls

def check_cross(x, y, gna=(), persp="global", filters=None, devices=None, vs_edges=True):
    cx, cy = x.shape[1], y.shape[1]
    full = ik.run_cross(x, y, gna, perspective=persp)
    filters = filters or filters_of(full)
    got = ik.run_cross_count_edges(x, y, gna, filters, devices=devices, perspective=persp)
    pi, pj = np.repeat(np.arange(cx), cy), np.tile(np.arange(cy), cx)
    for f, (t, a) in enumerate(filters):
        sel = mask(full, t, a)
        assert got["n_pass"][f] == int(sel.sum()), (f, t, a)
        assert np.array_equal(got["x_degree"][:, f], np.bincount(pi[sel], minlength=cx)), (f, t, a)
        assert np.array_equal(got["y_degree"][:, f], np.bincount(pj[sel], minlength=cy)), (f, t, a)
        if vs_edges and f % 7 == 0:
            e = ik.run_cross_edges(x, y, gna, min_abs_cor=t, max_pvalue=a, scale_max=False, perspective=persp)
            assert got["n_pass"][f] == e["i"].size
            assert np.array_equal(got["x_degree"][:, f], np.bincount(e["i"], minlength=cx))
            assert np.array_equal(got["y_degree"][:, f], np.bincount(e["j"], minlength=cy))
    assert np.array_equal(got["status_counts"], np.bincount(full["status"], minlength=_lib.NSTATUS)[:_lib.NSTATUS])
    assert bits(got["max_taumax"]) == bits(full["max_taumax"])
    return got


@pytest.mark.parametrize("persp", ["global", "local"])
@pytest.mark.parametrize("w", [1, 7, 4096, None])
def test_cross_against_pairs_and_edges(window, persp, w):
    window(w)
    n = 300 if w == 1 else 1200
    xy = degenerate_matrix(n, 50 if w == 1 else 130, seed=21)
    x, y = xy[:, :20 if w == 1 else 55], xy[:, 20 if w == 1 else 55:]
    check_cross(x, y, (), persp, vs_edges=w != 1)


def test_cross_csc_and_last_window(window):
    window(7)
    x = gen(1500, 40, "mixed", 0.05, seed=9)
    x[np.random.default_rng(9).random(x.shape) < 0.3] = 0.0
    y = gen(1500, 33, "ties", 0.05, seed=10)
    got = check_cross(sp.csc_matrix(x), y, GNA, vs_edges=False)
    dense = check_cross(x, y, GNA, filters=filters_of(ik.run_cross(x, y, GNA)), vs_edges=False)
    for k in ("n_pass", "x_degree", "y_degree", "status_counts"):
        assert np.array_equal(got[k], dense[k]), k
    rng = np.random.default_rng(3)
    a, b = rng.normal(size=(600, 30)), rng.normal(size=(600, 25))
    b[:, -1] = a[:, -1]  # the only pair with |raw| = 1 is the last of the cross order
    got = check_cross(np.asfortranarray(a), np.asfortranarray(b), filters=[(0.99, None), (0.99, 1e-300)])
    assert got["n_pass"][0] == 1 and got["x_degree"][-1, 0] == 1 and got["y_degree"][-1, 0] == 1


# ---------------------------------------------------------------- several devices

def device_lists():
    return [[0, 0], list(range(_lib.load().icikt_device_count()))]


@pytest.mark.parametrize("w", [7, None])
def test_multi_equals_one_device(window, w):
    window(w)
    x = degenerate_matrix(1500, 100, seed=31, kind="mixed")
    for diag in (False, True):
        f = filters_of(ik.run_pairs(x, (), include_diag=diag))
        one = ik.run_count_edges(x, (), f, include_diag=diag)
        for devs in device_lists():
            got = ik.run_count_edges(x, (), f, devices=devs, include_diag=diag)
            for k in ("n_pass", "degree", "status_counts"):
                assert np.array_equal(got[k], one[k]), (devs, k)
            assert bits(got["max_taumax"]) == bits(one["max_taumax"])
        csc = sp.csc_matrix(np.nan_to_num(x))
        one = ik.run_count_edges(csc, GNA, f, include_diag=diag)
        for devs in device_lists():
            got = ik.run_count_edges(csc, GNA, f, devices=devs, include_diag=diag)
            assert all(np.array_equal(got[k], one[k]) for k in ("n_pass", "degree", "status_counts")), devs
    x, y = x[:, :45], x[:, 45:]
    f = filters_of(ik.run_cross(x, y))
    one = ik.run_cross_count_edges(x, y, (), f)
    for devs in device_lists():
        got = ik.run_cross_count_edges(x, y, (), f, devices=devs)
        for k in ("n_pass", "x_degree", "y_degree", "status_counts"):
            assert np.array_equal(got[k], one[k]), (devs, k)
        assert bits(got["max_taumax"]) == bits(one["max_taumax"])


# ---------------------------------------------------------------- public API

TS, PS = [0.05, 0.2, 0.6], [None, 1e-3, 0.5]


@pytest.mark.parametrize("diag_good", [True, False])
@pytest.mark.parametrize("sparse", [False, True])
def test_api_matches_long_table(diag_good, sparse):
    x = gen(900, 40, "mixed", 0.1, seed=41)
    x[:, 2] = np.nan  # degenerate: warns, never an edge
    data = sp.csc_matrix(np.nan_to_num(x, nan=0.0)) if sparse else x
    names = [f"S{i}" for i in range(40)]
    got = ik.ici_kendalltau_edge_counts(data, min_abs_cor=TS, max_pvalue=PS, diag_good=diag_good, colnames=names)
    assert got["n_edges"].shape == (3, 3) and got["degree"].shape == (40, 3, 3) and got["names"] == names
    index = {s: k for k, s in enumerate(names)}
    for u, t in enumerate(TS):
        for v, p in enumerate(PS):
            tab = ik.ici_kendalltau(data, return_matrix=False, scale_max=False, min_abs_cor=t, max_pvalue=p,
                                    diag_good=diag_good, colnames=names)["cor"]
            s1 = np.array([index[s] for s in tab["s1"]], dtype=np.int64)
            s2 = np.array([index[s] for s in tab["s2"]], dtype=np.int64)
            assert got["n_edges"][u, v] == s1.size, (t, p)
            deg = np.bincount(s1, minlength=40) + np.bincount(s2[s1 != s2], minlength=40)
            assert np.array_equal(got["degree"][:, u, v], deg), (t, p)
    one = ik.ici_kendalltau_edge_counts(data, min_abs_cor=0.2, diag_good=diag_good, colnames=names)
    assert one["n_edges"].shape == () and one["n_edges"] == got["n_edges"][1, 2]
    ng = _lib.load().icikt_device_count()
    if ng > 1:
        every = ik.ici_kendalltau_edge_counts(data, min_abs_cor=0.2, diag_good=diag_good, colnames=names, n_gpus=ng)
        assert every["n_edges"] == one["n_edges"] and np.array_equal(every["degree"], one["degree"])


def test_api_warns_once_per_degenerate_class():
    x = degenerate_matrix(500, 12, seed=2)
    names = [f"S{i}" for i in range(12)]
    with pytest.warns(RuntimeWarning) as rec:
        ik.ici_kendalltau_edge_counts(x, min_abs_cor=[0.1, 0.3], colnames=names)
    texts = [str(w.message) for w in rec]
    assert sum("single unique value" in s for s in texts) == 1, texts


def test_cross_api_matches_long_table():
    xy = gen(900, 50, "ties", 0.1, seed=43)
    x, y = xy[:, :22], xy[:, 22:]
    xn, yn = [f"X{i}" for i in range(22)], [f"Y{i}" for i in range(28)]
    got = ik.ici_kendalltau_cross_edge_counts(x, y, min_abs_cor=TS, max_pvalue=PS, xnames=xn, ynames=yn)
    assert got["x_degree"].shape == (22, 3, 3) and got["y_degree"].shape == (28, 3, 3)
    for u, t in enumerate(TS):
        for v, p in enumerate(PS):
            tab = ik.ici_kendalltau_cross(x, y, return_matrix=False, scale_max=False, min_abs_cor=t, max_pvalue=p,
                                          xnames=xn, ynames=yn)["cor"]
            assert got["n_edges"][u, v] == len(tab["s1"]), (t, p)
            assert np.array_equal(got["x_degree"][:, u, v], [int(np.sum(tab["s1"] == s)) for s in xn])
            assert np.array_equal(got["y_degree"][:, u, v], [int(np.sum(tab["s2"] == s)) for s in yn])
    ng = _lib.load().icikt_device_count()
    if ng > 1:
        every = ik.ici_kendalltau_cross_edge_counts(x, y, min_abs_cor=TS, max_pvalue=PS, xnames=xn, ynames=yn, n_gpus=ng)
        assert np.array_equal(every["n_edges"], got["n_edges"]) and np.array_equal(every["x_degree"], got["x_degree"])
