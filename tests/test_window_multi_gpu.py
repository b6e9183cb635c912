"""The filtered and top-k all-pairs calls over several devices (icikt_all_pairs_edges_multi, icikt_all_pairs_topk_multi)
on the GPU.  Every result is compared bit for bit with the single-device call and with run_pairs masked (edges) or
sorted per column (top-k), with the helpers of test_edges_gpu.py and test_topk_gpu.py.

Repeated ordinals run the whole multi-device path on one GPU: sliced walks, the merge kernel and the host trim; with
two or more GPUs, list(range(ndev)) adds sharded K1 and real peer reads in the merge."""
import numpy as np
import pytest
import scipy.sparse as sp

import icikendalltau_b200 as ik
from icikendalltau_b200 import _lib
from tests import test_edges_gpu as E
from tests import test_topk_gpu as T
from tests.test_gpu_parity import gen

pytestmark = pytest.mark.gpu


def _ndev():
    return _lib.load().icikt_device_count()


def device_lists():
    nd = _ndev()
    lists = [[0, 0], [0] * 5, [0, 1 % max(nd, 1), 0]]
    if nd > 1:
        lists.append(list(range(nd)))
    return lists


DEVICE_LISTS = device_lists() if _ndev() > 0 else [[0, 0]]
IDS = ["-".join(map(str, d)) for d in DEVICE_LISTS]


def edges_grid(x, devices, what, gna=(), ts=E.T_BOUNDS, As=E.A_BOUNDS, include_diag=False, persps=("global", "local")):
    C = x.shape[1]
    for persp in persps:
        full = ik.run_pairs(x, gna, perspective=persp, include_diag=include_diag)
        for scale_max in (True, False):
            for t in ts:
                for a in As:
                    kw = dict(min_abs_cor=t, max_pvalue=a, scale_max=scale_max, perspective=persp,
                              include_diag=include_diag)
                    got = ik.run_edges(x, gna, devices=devices, **kw)
                    w = f"{what} {devices} {persp} scale_max={scale_max} t={t} a={a}"
                    E.same(got, ik.run_edges(x, gna, **kw), w + " vs one device")
                    E.same(got, E.expected(full, C, t, a, scale_max, include_diag), w)
                    E.same_max(got, full, w)


def topk_grid(x, devices, what, gna=(), ks=None, bys=("abs", "signed"), scales=(True, False),
              persps=("global", "local")):
    C = x.shape[1]
    pi, pj = T.pair_order(C)
    for persp in persps:
        full = ik.run_pairs(x, gna, perspective=persp)
        for k in ks or (1, 5, C - 1, C + 3):
            for by in bys:
                for scale_max in scales:
                    kw = dict(k=k, by=by, scale_max=scale_max, perspective=persp)
                    got = ik.run_topk(x, gna, devices=devices, **kw)
                    w = f"{what} {devices} {persp} k={k} by={by} scale_max={scale_max}"
                    T.same(got, ik.run_topk(x, gna, **kw), w + " vs one device")
                    T.same(got, T.topk_reference(C, k, by, scale_max, pi, pj, full, full["max_taumax"]), w)
                    T.same_max(got, full["max_taumax"], w)


@pytest.mark.parametrize("devices", DEVICE_LISTS, ids=IDS)
def test_edges_multi_equal_one_device(devices):
    x = gen(2000, 120, "mixed", 0.1, seed=51)
    edges_grid(x, devices, "2000x120")


@pytest.mark.parametrize("devices", DEVICE_LISTS, ids=IDS)
def test_topk_multi_equal_one_device(devices):
    x = gen(2000, 120, "ties", 0.1, seed=52)
    topk_grid(x, devices, "2000x120")


@pytest.mark.parametrize("window", [1, 7, 4096])
def test_small_windows(monkeypatch, window):
    """windows (and slices) that cut units and rows mid-way"""
    monkeypatch.setenv("ICIKT_EDGE_WINDOW", str(window))
    n, C = (300, 30) if window == 1 else (2000, 120)
    x = gen(n, C, "mixed", 0.15, seed=60 + window)
    for devices in ([0, 0, 0], DEVICE_LISTS[-1]):
        edges_grid(x, devices, f"window={window}", ts=(None, 0.3), As=(None, 1e-3), include_diag=window == 7,
                   persps=("global",))
        topk_grid(x, devices, f"window={window}", ks=(1, 5, C - 1), scales=(True,), persps=("global",))
    edges_grid(x, [0] * 5, f"window={window}", ts=(0.5,), As=(None,), persps=("local",))
    topk_grid(x, [0] * 5, f"window={window}", ks=(3,), bys=("abs",), scales=(False,), persps=("local",))


@pytest.mark.parametrize("window", [7, None])
@pytest.mark.parametrize("devices", [[0, 0, 0], None], ids=["0-0-0", "all"])
def test_late_maximum_in_the_last_slice(monkeypatch, window, devices):
    """the largest taumax is the last pair: only the last device sees it, so the rows the earlier devices hold
    against their own maximum must be trimmed by the final one"""
    if window:
        monkeypatch.setenv("ICIKT_EDGE_WINDOW", str(window))
    devices = devices or DEVICE_LISTS[-1]
    n, C = 1500, 100
    x = E.late_maximum_matrix(n, C, seed=3)
    ptot = C * (C - 1) // 2
    last_lo = ptot * (len(devices) - 1) // len(devices)
    for persp in ("global", "local"):
        full = ik.run_pairs(x, (), perspective=persp)
        tm = full["taumax"]
        assert np.nanargmax(tm) == tm.size - 1 and np.nanmax(tm[:last_lo]) < tm[-1]
        t = float(np.quantile(np.abs(full["raw"][full["status"] == 0]), 0.9))
        early = (full["status"] == 0) & (np.abs(full["raw"]) >= t * np.nanmax(tm[:last_lo]))
        early &= np.abs(full["raw"] / tm[-1]) < t
        assert early[:last_lo].sum() > 0  # rows an earlier device holds that the final maximum removes
        for a in (None, 1e-3):
            got = ik.run_edges(x, (), min_abs_cor=t, max_pvalue=a, perspective=persp, devices=devices)
            E.same(got, E.expected(full, C, t, a, True), f"late maximum {persp} {devices} window={window} a={a}")
            E.same_max(got, full, "late maximum")
        topk_grid(x, devices, "late maximum", ks=(4,), bys=("abs",), persps=(persp,))


def test_duplicated_columns_tie_across_slices():
    """identical and negated columns: equal keys come from different slices and the partner decides"""
    rng = np.random.default_rng(21)
    base = rng.normal(size=(400, 6))
    x = np.asfortranarray(base[:, rng.integers(0, 6, size=90)])
    x[:, 40:50] = -x[:, 40:50]
    for devices in ([0, 0, 0], [0] * 5, DEVICE_LISTS[-1]):
        topk_grid(x, devices, "duplicated", ks=(1, 4, 17, 89), persps=("global",))
        edges_grid(x, devices, "duplicated", ts=(0.5,), As=(None,), persps=("global",))


def test_full_lists_at_k_max():
    C = 1100
    x = gen(800, C, "normal", 0.05, seed=41)
    for devices in ([0, 0], DEVICE_LISTS[-1]):
        topk_grid(x, devices, "k=1024", ks=(_lib.TOPK_MAX,), scales=(True,), persps=("global",))
    got = ik.run_topk(x, (), k=_lib.TOPK_MAX, devices=[0, 0, 0])
    assert (got["n_neighbors"] == _lib.TOPK_MAX).all()


def test_include_diag_edges():
    x = gen(1000, 40, "normal", 0.1, seed=9)
    for devices in ([0, 0, 0], DEVICE_LISTS[-1]):
        edges_grid(x, devices, "include_diag", ts=(None, 0.0, 0.2), As=(None,), include_diag=True, persps=("global",))


@pytest.mark.parametrize("C,devices", [(1, [0, 0]), (2, [0, 0, 0]), (3, [0] * 5), (4, [0] * 16)])
def test_degenerate_sizes(C, devices):
    """C = 1, empty slices (C = 2 on three devices) and empty column blocks (C < n_devices)"""
    x = np.asfortranarray(np.random.default_rng(C).normal(size=(50, C)))
    for include_diag in (False, True):
        for t in (None, 0.0):
            kw = dict(min_abs_cor=t, max_pvalue=None if t is not None else 1.0, include_diag=include_diag)
            got = ik.run_edges(x, (), devices=devices, **kw)
            want = ik.run_edges(x, (), **kw)
            E.same(got, want, f"C={C} {devices} {kw}")
            assert np.array_equal(np.float64(got["max_taumax"]).view(np.int64),
                                  np.float64(want["max_taumax"]).view(np.int64))
    for k in (1, 3, 7):
        for by in ("abs", "signed"):
            got = ik.run_topk(x, (), k=k, by=by, devices=devices)
            want = ik.run_topk(x, (), k=k, by=by)
            T.same(got, want, f"C={C} {devices} k={k}")
            T.same_max(got, want["max_taumax"], f"C={C}")


def test_csc_twins_equal_dense():
    rng = np.random.default_rng(6)
    d = rng.normal(size=(3000, 80)) + rng.normal(size=(3000, 1))
    d[rng.random(d.shape) < 0.5] = 0.0
    a = sp.csc_matrix(d)
    dense = np.asfortranarray(d)
    gna = (np.nan, np.inf, 0.0)
    for devices in ([0, 0, 0], DEVICE_LISTS[-1]):
        for t, al in ((0.2, None), (None, 1e-2)):
            x = ik.run_edges(a, gna, min_abs_cor=t, max_pvalue=al, devices=devices)
            E.same(x, ik.run_edges(dense, gna, min_abs_cor=t, max_pvalue=al, devices=devices), f"csc {devices} t={t}")
            E.same(x, ik.run_edges(dense, gna, min_abs_cor=t, max_pvalue=al), f"csc {devices} vs one device")
        for k, by in ((7, "abs"), (79, "signed")):
            x = ik.run_topk(a, gna, k=k, by=by, devices=devices)
            T.same(x, ik.run_topk(dense, gna, k=k, by=by, devices=devices), f"csc {devices} k={k}")
            T.same(x, ik.run_topk(dense, gna, k=k, by=by), f"csc {devices} k={k} vs one device")


def test_long_vectors_in_place_on_two_devices():
    n, C = 60000, 24
    assert _lib.launch_shape(n)["variant"] == "inplace"
    x = gen(n, C, "ties", 0.1, seed=n + C)
    devices = [0, 1 % max(_ndev(), 1)]
    edges_grid(x, devices, "60000x24", ts=(None, 0.3), As=(None, 1e-3), persps=("global",))
    topk_grid(x, devices, "60000x24", ks=(1, 5, 23), scales=(True,), persps=("global",))


def test_max_edges_without_scale_max():
    """held rows are final rows: the limit fails exactly when more pairs pass, and the next call succeeds"""
    x = gen(2000, 100, "normal", 0.0, seed=10)
    full = ik.run_pairs(x, ())
    want = E.expected(full, 100, 0.3, None, False)
    m = want["i"].size
    assert m > 10
    for devices in ([0, 0, 0], DEVICE_LISTS[-1]):
        E.same(ik.run_edges(x, (), min_abs_cor=0.3, scale_max=False, max_edges=m, devices=devices), want, "limit = count")
        with pytest.raises(ik.IciktError) as e:
            ik.run_edges(x, (), min_abs_cor=0.3, scale_max=False, max_edges=m - 1, devices=devices)
        assert e.value.code == _lib.ERR_LIMIT
        E.same(ik.run_edges(x, (), min_abs_cor=0.3, scale_max=False, devices=devices), want, "after the limit")
    # a p-value bound alone is exact too, with scale_max
    want = E.expected(full, 100, None, 1e-3, True)
    m = want["i"].size
    with pytest.raises(ik.IciktError) as e:
        ik.run_edges(x, (), max_pvalue=1e-3, max_edges=m - 1, devices=[0, 0])
    assert e.value.code == _lib.ERR_LIMIT
    E.same(ik.run_edges(x, (), max_pvalue=1e-3, max_edges=m, devices=[0, 0]), want, "p-value limit = count")


def test_interleaved_calls_keep_their_results():
    """the multi-device window plans, the single-device window plan, the per-pair multi plans and the per-pair plan of
    one device (the single-device call and devices=[0], alternated) do not disturb each other"""
    x = gen(1500, 90, "mixed", 0.1, seed=71)
    devices = DEVICE_LISTS[-1]
    e0 = ik.run_edges(x, (), min_abs_cor=0.3, devices=devices)
    k0 = ik.run_topk(x, (), k=6, devices=devices)
    s0 = ik.run_edges(x, (), min_abs_cor=0.3)
    p0 = ik.run_pairs(x, (), devices=devices)
    m0 = _lib.run_matrices(x, (), devices=devices)
    s1 = ik.run_pairs(x, ())
    for _ in range(2):
        for one in ([0], None):
            p = ik.run_pairs(x, (), devices=one)
            for key in ("raw", "pvalue", "taumax", "completeness", "status"):
                assert np.array_equal(p[key].view(np.uint8), s1[key].view(np.uint8)), (one, key)
        E.same(ik.run_edges(x, (), min_abs_cor=0.3, devices=devices), e0, "multi edges again")
        T.same(ik.run_topk(x, (), k=6, devices=devices), k0, "multi top-k again")
        E.same(ik.run_edges(x, (), min_abs_cor=0.3), s0, "single edges again")
        p = ik.run_pairs(x, (), devices=devices)
        for key in ("raw", "pvalue", "taumax", "completeness", "status"):
            assert np.array_equal(p[key].view(np.uint8), p0[key].view(np.uint8)), key
        m = _lib.run_matrices(x, (), devices=devices)
        for key in _lib.MATRIX_NAMES:
            assert np.array_equal(m[key].view(np.int64), m0[key].view(np.int64)), key
    E.same(e0, s0, "multi vs single")
    _lib.release_workspace()
    E.same(ik.run_edges(x, (), min_abs_cor=0.3, devices=devices), e0, "after release_workspace")
    T.same(ik.run_topk(x, (), k=6, devices=devices), k0, "after release_workspace")


def test_ici_kendalltau_topk_n_gpus():
    x = gen(1500, 30, "mixed", 0.1, seed=12)
    names = [f"s{k}" for k in range(30)]
    one = ik.ici_kendalltau_topk(x, 4, colnames=names)
    many = ik.ici_kendalltau_topk(x, 4, colnames=names, n_gpus=max(2, _ndev()) if _ndev() > 1 else 1)
    T.same(many, one, "n_gpus")
    assert many["neighbors"].tolist() == one["neighbors"].tolist()
    got = ik.run_topk(x, (np.nan, np.inf, 0.0), k=4, devices=[0, 0])
    T.same(got, one, "repeated ordinals")


def test_timings_and_launches():
    x = gen(2000, 200, "normal", 0.1, seed=13)
    got = ik.run_edges(x, (), min_abs_cor=0.3, devices=[0, 0])
    one = ik.run_edges(x, (), min_abs_cor=0.3)
    assert got["timings"]["pairs_ms"] > 0 and got["timings"]["total_ms"] > 0
    assert got["timings"]["n_launches"] > one["timings"]["n_launches"]  # summed over the devices
    got = ik.run_topk(x, (), k=8, devices=[0, 0])
    assert got["timings"]["pairs_ms"] > 0 and got["timings"]["d2h_ms"] > 0
