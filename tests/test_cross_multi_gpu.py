"""The cross calls over several devices (icikt_cross_pairs_multi, icikt_cross_edges_multi, icikt_cross_topk_multi) on
the GPU.  Every result is compared bit for bit with the single-device cross call and with icikt_pair_list on [X | Y]
(the helpers of test_cross_gpu.py).

Repeated ordinals run the whole multi-device path on one GPU: sliced walks, the merge kernel across the two sides and
the host join.  ICIKT_FORCE_PEER_GATHER=1 makes repeated ordinals take the sharded column phase too (K1 on a share of
[X | Y] per worker, then the gather of the tables), which one GPU otherwise never runs; with two or more GPUs,
list(range(ndev)) adds it between distinct devices with real peer reads."""
import numpy as np
import pytest
import scipy.sparse as sp

import icikendalltau_b200 as ik
from icikendalltau_b200 import _lib
from tests.test_cross_gpu import (FIELDS, bits, degenerate_pair, dense, host_lists, masked, reference, same_edges,
                                  same_lists, same_pairs, window)  # noqa: F401 (window: fixture)
from tests.test_edges_gpu import late_maximum_matrix
from tests.test_gpu_parity import gen
from tests.test_launch_variants_gpu import device_stats, tier2_matrix, tier_of
from tests.test_window_multi_gpu import DEVICE_LISTS, IDS

pytestmark = pytest.mark.gpu


@pytest.fixture
def gather(monkeypatch):
    monkeypatch.setenv("ICIKT_FORCE_PEER_GATHER", "1")


def pairs_both(x, y, devices, what, gna=(), **kw):
    got = ik.run_cross(x, y, gna, devices=devices, **kw)
    same_pairs(got, ik.run_cross(x, y, gna, **kw), what + " vs one device")
    lo, hi = kw.get("pair_lo", 0), kw.get("pair_hi", 0)
    if hi > lo or hi == 0:
        same_pairs(got, reference(x, y, gna, lo, hi or None, **{k: v for k, v in kw.items()
                                                               if k not in ("pair_lo", "pair_hi")}), what)
    return got


def edges_both(x, y, devices, what, t, a, scale_max, gna=(), full=None, **kw):
    got = _lib.run_cross_edges(x, y, gna, t, a, scale_max, devices=devices, **kw)
    same_edges(got, _lib.run_cross_edges(x, y, gna, t, a, scale_max, **kw), what + " vs one device")
    assert bits(got["max_taumax"]) == bits(full["max_taumax"]), what
    same_edges(got, masked(full, dense(x).shape[1], dense(y).shape[1], t, a, scale_max), what)


def topk_both(x, y, devices, what, k, by, scale_max, side, gna=(), full=None, **kw):
    cx, cy = dense(x).shape[1], dense(y).shape[1]
    got = _lib.run_cross_topk(x, y, gna, k, by, scale_max, side, devices=devices, **kw)
    one = _lib.run_cross_topk(x, y, gna, k, by, scale_max, side, **kw)
    assert bits(got["max_taumax"]) == bits(one["max_taumax"]) == bits(full["max_taumax"]), what
    for s in ("x", "y"):
        key = s + "_side"
        assert (key in got) == (key in one) == (side in (s, "both")), what
        if key in got:
            same_lists(got[key], one[key], f"{what}: {s} side vs one device")
            same_lists(got[key], host_lists(full, cx, cy, k, by, scale_max, s), f"{what}: {s} side")


# ---------------------------------------------------------------- icikt_cross_pairs_multi
@pytest.mark.parametrize("devices", DEVICE_LISTS, ids=IDS)
@pytest.mark.parametrize("w", [1, 7, 4096])
def test_pairs_multi(window, w, devices):
    window(w)
    x, y = degenerate_pair(seed=w + 3)
    for persp in ("global", "local"):
        for alt, cont in (("two.sided", False), ("less", True), ("greater", False)):
            got = pairs_both(x, y, devices, f"{devices} {persp} {alt} continuity={cont} window={w}", (np.nan,),
                             perspective=persp, alternative=alt, continuity=cont)
            assert (got["status"] != 0).sum() > 0


@pytest.mark.parametrize("lo,hi", [(0, 1), (3, 4), (29, 30), (17, 17), (5, 29), (0, 30), (0, 0)])
def test_pair_slices_multi(window, lo, hi):
    """a slice of the cross order over 5 workers: 1 pair leaves four of them none, (17, 17) is empty"""
    window(7)
    x, y = degenerate_pair(seed=5)
    for devices in ([0] * 5, [0, 0]):
        got = pairs_both(x, y, devices, f"{devices} [{lo}, {hi})", pair_lo=lo, pair_hi=hi)
        assert got["raw"].size == (hi - lo if hi else 30)
        if hi == lo and hi:
            assert np.isnan(got["max_taumax"])


def test_all_degenerate_is_nan(window):
    window(3)
    x = np.full((50, 3), 2.0)
    y = np.asfortranarray(np.column_stack([np.full(50, np.nan), np.arange(50.0), np.arange(50.0)]))
    got = ik.run_cross(x, y, (), devices=[0, 0, 0])
    same_pairs(got, ik.run_cross(x, y, ()), "every pair degenerate")
    assert np.isnan(got["max_taumax"]) and (got["status"] != 0).all()


# ---------------------------------------------------------------- icikt_cross_edges_multi
@pytest.mark.parametrize("devices", DEVICE_LISTS, ids=IDS)
@pytest.mark.parametrize("w", [1, 7, 4096])
def test_edges_multi(window, w, devices):
    window(w)
    x, y = degenerate_pair(seed=11, cx=7, cy=9)
    for persp in ("global", "local"):
        full = reference(x, y, (), perspective=persp)
        for scale_max in (True, False):
            for t, a in ((None, None), (0.3, None), (None, 1e-2), (0.5, 1e-3), (1.01, None)):
                edges_both(x, y, devices, f"{devices} {persp} window={w} scale_max={scale_max} t={t} a={a}", t, a,
                           scale_max, full=full, perspective=persp)


@pytest.mark.parametrize("devices", DEVICE_LISTS, ids=IDS)
def test_edges_multi_late_maximum_and_limit(window, devices):
    """the pair of largest taumax is the last pair of the cross order, so only the last slice holds the maximum"""
    window(7)
    m = late_maximum_matrix(800, 24, seed=3)
    x = np.asfortranarray(np.column_stack([m[:, :11], m[:, 22]]))
    y = np.asfortranarray(np.column_stack([m[:, 11:22], m[:, 23]]))
    cx, cy = x.shape[1], y.shape[1]
    full = reference(x, y, ())
    tm = full["taumax"]
    assert np.nanargmax(tm) == tm.size - 1 and tm[-1] == 1.0
    t = float(np.quantile(np.abs(full["raw"][full["status"] == 0]), 0.8))
    edges_both(x, y, devices, f"{devices} late maximum", t, None, True, full=full)
    # without scale_max the rows held are the final ones in every window: max_edges is exact
    want = masked(full, cx, cy, t, None, False)
    m_pass = want["i"].size
    assert m_pass > 1
    same_edges(_lib.run_cross_edges(x, y, (), t, None, False, max_edges=m_pass, devices=devices), want,
               f"{devices} max_edges = count")
    with pytest.raises(ik.IciktError) as e:
        _lib.run_cross_edges(x, y, (), t, None, False, max_edges=m_pass - 1, devices=devices)
    assert e.value.code == _lib.ERR_LIMIT
    same_edges(_lib.run_cross_edges(x, y, (), t, None, False, devices=devices), want, f"{devices} after the limit")


# ---------------------------------------------------------------- icikt_cross_topk_multi
@pytest.mark.parametrize("devices", DEVICE_LISTS, ids=IDS)
def test_topk_multi(window, devices):
    window(7)
    x, y = degenerate_pair(seed=21, cx=6, cy=9)
    x[:, 5] = np.round(x[:, 5])  # equal raws with different partners
    y[:, 6] = np.round(y[:, 6])
    full = reference(x, y, ())
    for side in ("x", "y", "both"):
        other = 9 if side == "x" else 6
        for k in (1, 5, other + 1):
            for by in ("abs", "signed"):
                for scale_max in (True, False):
                    topk_both(x, y, devices, f"{devices} side={side} k={k} by={by} scale_max={scale_max}", k, by,
                              scale_max, side, full=full)


def test_topk_multi_k_1024(window):
    window(None)
    m = gen(200, 3 + 1100, "ties", 0.05, 31)
    x, y = m[:, :3], m[:, 3:]
    full = reference(x, y, ())
    for devices in ([0, 0], [0] * 5):
        topk_both(x, y, devices, f"{devices} k=1024", 1024, "abs", False, "both", full=full)
        topk_both(x, y, devices, f"{devices} k=1024", 1024, "signed", True, "x", full=full)


@pytest.mark.parametrize("cx,cy", [(1, 9), (9, 1), (1, 1), (2, 2)])
def test_topk_multi_narrow(window, cx, cy):
    """one-column sides, and Cx * Cy below the number of devices"""
    window(1)
    m = gen(300, cx + cy, "ties", 0.05, cx * 10 + cy)
    x, y = m[:, :cx], m[:, cx:]
    full = reference(x, y, ())
    for devices in ([0] * 5, [0, 0]):
        for side in ("x", "y", "both"):
            topk_both(x, y, devices, f"{devices} {cx}x{cy} side={side}", 3, "abs", True, side, full=full)
        pairs_both(x, y, devices, f"{devices} {cx}x{cy}")
        edges_both(x, y, devices, f"{devices} {cx}x{cy}", 0.1, None, True, full=full)


# ---------------------------------------------------------------- the sharded column phase
@pytest.mark.parametrize("form", ["dense-dense", "csc-dense", "dense-csc", "csc-csc"])
def test_gathered_columns_dense_and_csc(window, gather, form):
    """shares of [X | Y] that straddle column Cx (7): [0, 8) and [8, 16) over two workers, [0, 5), [5, 10), [10, 16)
    over three; both sides CSC must expand X's part before Y's part overwrites the CSC buffers"""
    a = sp.random(500, 7, density=0.3, format="csc", random_state=1)
    b = sp.random(500, 9, density=0.5, format="csc", random_state=2)
    a.data = np.round(a.data * 5)
    x = a if form.startswith("csc") else dense(a)
    y = b if form.endswith("csc") else dense(b)
    gna = (np.nan, np.inf, 0.0)
    full = reference(x, y, gna)
    for w in (7, 4096):
        window(w)
        for devices in ([0, 0], [0, 0, 0], [0] * 5):
            what = f"{form} {devices} window={w}"
            pairs_both(x, y, devices, what, gna)
            edges_both(x, y, devices, what, 0.2, None, True, gna, full=full)
            topk_both(x, y, devices, what, 4, "abs", True, "both", gna, full=full)


def test_gathered_tier_from_y(window, gather):
    """Y is a tier-2 matrix and X tier 0: over three workers, the first one's share of [X | Y] ([0, 5) of 15) holds
    X's columns only, and it gets the tier from the gathered statistics"""
    window(None)
    y = tier2_matrix(4096, 17, 200, seed=3)[1]
    x = np.asfortranarray(np.random.default_rng(7).standard_normal((4096, 6)))
    assert tier_of(device_stats(x), 4096) == 0
    assert tier_of(device_stats(y), 4096) == 2
    full = reference(x, y, ())
    for devices in ([0, 0], [0, 0, 0]):
        for persp in ("global", "local"):
            pairs_both(x, y, devices, f"tier 2 in y {devices} {persp}", perspective=persp)
        topk_both(x, y, devices, f"tier 2 in y {devices}", 2, "abs", True, "both", full=full)


# ---------------------------------------------------------------- calls that share the worker plan slots
def test_interleaved_calls(window):
    window(7)
    x, y = degenerate_pair(seed=61, cx=6, cy=8)
    full = reference(x, y, ())
    z = gen(600, 20, "mixed", 0.1, seed=62)
    for devices in ([0, 0, 0], [0] * 5):
        same_pairs(ik.run_cross(x, y, ()), full, "single")
        same_pairs(ik.run_cross(x, y, (), devices=devices), full, f"{devices} multi")
        got = ik.run_edges(z, (), min_abs_cor=0.3, devices=devices)
        same_edges(got, ik.run_edges(z, (), min_abs_cor=0.3), f"{devices} all-pairs edges")
        topk_both(x, y, devices, f"{devices} after the all-pairs call", 3, "signed", False, "both", full=full)
        same_pairs(ik.run_cross(x, y, (), devices=devices), full, f"{devices} multi again")
