"""The filtered and top-k all-pairs calls over several devices without a GPU: the argument checks of the four
entry points (icikt_all_pairs_edges_multi, icikt_all_pairs_topk_multi and their CSC twins) that run before any
device is touched, the device merge of the top-k lists (compiled for the host from the header the merge kernel
uses) against NumPy's lexsort, and the Python routing with a stand-in for the library."""
import ctypes
import os
import subprocess

import numpy as np
import pytest
import scipy.sparse as sp

import icikendalltau_b200 as ik
from icikendalltau_b200 import _lib

HERE = os.path.dirname(os.path.abspath(__file__))
NAN = float("nan")


# ---------------------------------------------------------------- refusals before any device work

def _lead(name, n, C, unsorted=False):
    """(leading arguments, the objects they point into) of a dense or CSC entry point"""
    if not name.endswith("_csc"):
        x = np.asfortranarray(np.random.default_rng(0).normal(size=(n, max(C, 1))))
        return (x.ctypes.data, n, C, n), [x]
    a = sp.random(n, max(C, 1), density=0.5, format="csc", random_state=1)
    m = _lib.CSC(a)
    if unsorted:  # swap the first two rows of the first column with two entries
        c = int(np.nonzero(np.diff(m.colptr) >= 2)[0][0])
        s = int(m.colptr[c])
        m.rowidx[s], m.rowidx[s + 1] = m.rowidx[s + 1], m.rowidx[s]
    return (m.colptr.ctypes.data, m.rowidx.ctypes.data, m.values.ctypes.data, n, C), [m]


def _edges(name, opts=None, n_devices=2, devices=None, filter_=True, out=True, max_edges=0, n=20, C=5,
           unsorted=False):
    L = _lib.load()
    lead, keep = _lead(name, n, C, unsorted)
    o = opts if opts is not None else _lib.make_opts()
    dev = None if devices is None else np.ascontiguousarray(devices, dtype=np.int32)
    f = _lib.EdgeFilter(0.5, NAN, 1, 0, max_edges)
    h = ctypes.c_void_p(12345)
    rc = getattr(L, name)(*lead, None, 0, ctypes.byref(o), None if dev is None else dev.ctypes.data, n_devices,
                          ctypes.byref(f) if filter_ else None, ctypes.byref(h) if out else None, None, None)
    msg = L.icikt_last_error().decode()
    if rc == _lib.OK:
        L.icikt_edges_free(h)
    return rc, msg, h.value


def _topk(name, opts=None, n_devices=2, devices=None, k=4, by=0, index=True, n=20, C=5, unsorted=False):
    L = _lib.load()
    lead, keep = _lead(name, n, C, unsorted)
    o = opts if opts is not None else _lib.make_opts()
    dev = None if devices is None else np.ascontiguousarray(devices, dtype=np.int32)
    idx = np.full((max(C, 1), max(k, 1)), 7, dtype=np.int32)
    rc = getattr(L, name)(*lead, None, 0, ctypes.byref(o), None if dev is None else dev.ctypes.data, n_devices, k,
                          by, 1, idx.ctypes.data if index else None, None, None, None, None, None, None, None, None)
    return rc, L.icikt_last_error().decode(), idx


COMMON = {  # (opts, call arguments, words of the message)
    "n_devices_zero": ({}, dict(n_devices=0), "n_devices"),
    "n_devices_17": ({}, dict(n_devices=17, devices=[0] * 17), "n_devices"),
    "n_devices_negative": ({}, dict(n_devices=-1), "n_devices"),
    "pair_lo": (dict(pair_lo=1, pair_hi=5), {}, "pair_lo"),
    "complete": (dict(perspective="complete"), {}, "perspective"),
    "naive": (dict(kernel=_lib.KERNEL_NAIVE), {}, "tiled kernel"),
    "want_counts": (dict(want_counts=True), {}, "want_counts"),
    "n_zero": ({}, dict(n=0), ">= 1"),
    "C_zero": ({}, dict(C=0), ">= 1"),
}
EDGES = dict(COMMON, **{
    "null_filter": ({}, dict(filter_=False), "filter is NULL"),
    "null_out": ({}, dict(out=False), "out is NULL"),
    "max_edges_negative": ({}, dict(max_edges=-1), "max_edges"),
})
TOPK = dict(COMMON, **{
    "k_zero": ({}, dict(k=0), "k must be"),
    "k_above_max": ({}, dict(k=1025), "k must be"),
    "by_two": ({}, dict(by=2), "by must be"),
    "null_index": ({}, dict(index=False), "index is NULL"),
    "include_diag": (dict(include_diag=True), {}, "include_diag"),
})


@pytest.mark.parametrize("case", sorted(EDGES))
@pytest.mark.parametrize("name", ["icikt_all_pairs_edges_multi", "icikt_all_pairs_edges_multi_csc"])
def test_edges_multi_refused_before_any_device_work(name, case):
    okw, ckw, words = EDGES[case]
    if name.endswith("_csc") and case in ("n_zero", "C_zero"):
        words = ""  # the CSC checks speak first
    rc, msg, h = _edges(name, opts=_lib.make_opts(**okw), **ckw)
    assert rc == _lib.ERR_BAD_ARG, (rc, msg)
    assert words in msg, msg
    if case != "null_out":
        assert h is None  # *out is cleared, nothing allocated


@pytest.mark.parametrize("case", sorted(TOPK))
@pytest.mark.parametrize("name", ["icikt_all_pairs_topk_multi", "icikt_all_pairs_topk_multi_csc"])
def test_topk_multi_refused_before_any_device_work(name, case):
    okw, ckw, words = TOPK[case]
    if name.endswith("_csc") and case in ("n_zero", "C_zero"):
        words = ""
    rc, msg, idx = _topk(name, opts=_lib.make_opts(**okw), **ckw)
    assert rc == _lib.ERR_BAD_ARG, (rc, msg)
    assert words in msg, msg
    assert (idx == 7).all()  # nothing written


def test_unsorted_csc_column_is_refused():
    rc, msg, h = _edges("icikt_all_pairs_edges_multi_csc", unsorted=True)
    assert rc == _lib.ERR_BAD_ARG and "column" in msg, msg
    assert h is None
    rc, msg, idx = _topk("icikt_all_pairs_topk_multi_csc", unsorted=True)
    assert rc == _lib.ERR_BAD_ARG and "column" in msg, msg
    assert (idx == 7).all()


def test_sixteen_devices_pass_the_checks():
    """n_devices = 16 is the upper limit: the call gets past the argument checks (to the device, or to
    ERR_NO_DEVICE without one)"""
    for call, name in ((_edges, "icikt_all_pairs_edges_multi"), (_topk, "icikt_all_pairs_topk_multi")):
        rc, msg, _ = call(name, n_devices=16, devices=[0] * 16)
        assert rc != _lib.ERR_BAD_ARG or "n_devices" not in msg, msg


# ---------------------------------------------------------------- the device merge

@pytest.fixture(scope="module")
def host(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("merge") / "libtopk_merge_host.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-x", "c++",
                           os.path.join(HERE, "topk_merge_host.cpp"), "-o", out])
    L = ctypes.CDLL(out)
    vp = ctypes.c_void_p
    L.topk_merge_host.argtypes = [ctypes.c_int, vp, vp, vp, ctypes.c_int, ctypes.c_int, vp, vp]
    L.topk_merge_host.restype = ctypes.c_int
    return L


def _order(raw, partner, by):
    return np.lexsort((partner, -np.abs(raw) if by == 0 else -raw))


def _check_merge(host, raw, partner, owner, n_dev, k, by):
    """device d holds the top k of the candidates it owns; the merge of those lists must be the top k of all"""
    lists = []
    for d in range(n_dev):
        sel = np.nonzero(owner == d)[0]
        lists.append(sel[_order(raw[sel], partner[sel], by)][:k])
    off = np.zeros(n_dev + 1, dtype=np.int64)
    off[1:] = np.cumsum([len(li) for li in lists])
    cat = np.concatenate(lists).astype(np.int64) if off[-1] else np.zeros(0, dtype=np.int64)
    lraw = np.ascontiguousarray(raw[cat], dtype=np.float64)
    lpart = np.ascontiguousarray(partner[cat], dtype=np.int32)
    out_part = np.full(k, -9, dtype=np.int32)
    out_src = np.full(k, -9, dtype=np.int32)
    a = host.topk_merge_host(n_dev, off.ctypes.data, lraw.ctypes.data, lpart.ctypes.data, k, by,
                             out_part.ctypes.data, out_src.ctypes.data)
    want = _order(raw, partner, by)[:k]
    assert a == want.size
    assert np.array_equal(out_part[:a], partner[want])
    d, pos = out_src[:a] // 1024, out_src[:a] % 1024
    assert np.array_equal(lpart[off[d] + pos], out_part[:a])  # the source holds that entry
    assert np.array_equal(lraw[off[d] + pos].view(np.int64), raw[want].view(np.int64))


@pytest.mark.parametrize("by", [0, 1])
def test_merge_of_random_lists_equals_lexsort(host, by):
    rng = np.random.default_rng(7 + by)
    for trial in range(300):
        n_dev = int(rng.integers(2, 17))
        k = int(rng.choice([1, 2, 3, 5, 16, 31, 64, 100, 257, 1024]))
        m = int(rng.integers(0, 3 * k + 2 * n_dev))
        raw = rng.uniform(-1, 1, size=m)
        if trial % 3 == 0:  # many equal keys across the lists: the partner decides
            raw = rng.choice([0.5, -0.5, 0.25, -0.25, 0.0, -0.0, 1.0], size=m)
        partner = rng.permutation(max(m, 1) * 3)[:m].astype(np.int32)
        owner = rng.integers(0, n_dev, size=m)
        _check_merge(host, raw, partner, owner, n_dev, k, by)


@pytest.mark.parametrize("by", [0, 1])
def test_merge_equal_keys_in_every_list(host, by):
    """one value everywhere: the merged list is the k smallest partners, taken from every device"""
    for n_dev, k in ((2, 1), (3, 7), (16, 1024), (16, 5)):
        m = 4000
        raw = np.full(m, -0.75)
        partner = np.random.default_rng(k).permutation(m).astype(np.int32)
        owner = np.arange(m) % n_dev
        _check_merge(host, raw, partner, owner, n_dev, k, by)


def test_merge_lists_shorter_than_k(host):
    rng = np.random.default_rng(3)
    for n_dev in (2, 5, 16):
        for k in (1024, 40):
            m = k // 2
            raw = rng.normal(size=m)
            partner = rng.permutation(m).astype(np.int32)
            owner = rng.integers(0, n_dev, size=m)
            owner[owner == 1] = 0  # device 1 holds nothing
            _check_merge(host, raw, partner, owner, n_dev, k, 0)


def test_merge_full_lists_from_every_device(host):
    rng = np.random.default_rng(4)
    n_dev, k = 16, 1024
    m = n_dev * k
    raw = np.round(rng.uniform(-1, 1, size=m) * 200) / 200
    partner = rng.permutation(m).astype(np.int32)
    owner = np.repeat(np.arange(n_dev), k)
    _check_merge(host, raw, partner, owner, n_dev, k, 1)


# ---------------------------------------------------------------- Python routing

def _stub(monkeypatch, calls):
    """stand-ins for the filtered calls that record their name and the devices they were handed"""
    real = _lib.load()

    def call(name):
        def f(*args):
            at = 5 if name.endswith("_csc") else 4  # global_na
            rec = dict(name=name, C=args[at - 1] if name.endswith("_csc") else args[2])
            if "multi" in name:
                dev, ndev = args[at + 3], args[at + 4]
                rec["devices"] = list((ctypes.c_int32 * ndev).from_address(dev)) if ndev else []
            if "topk" in name:  # every list empty
                k, index = args[at + (5 if "multi" in name else 3)], args[at + (8 if "multi" in name else 6)]
                (ctypes.c_int32 * (rec["C"] * k)).from_address(index)[:] = [-1] * (rec["C"] * k)
            calls.append(rec)
            return 0
        return f

    class Stub:
        def __getattr__(self, name):
            if name.startswith(("icikt_all_pairs_edges", "icikt_all_pairs_topk")):
                return call(name)
            if name == "icikt_edges_count":
                return lambda h: 0
            if name == "icikt_edges_copy":
                return lambda *a: 0
            if name == "icikt_edges_free":
                return lambda h: None
            return getattr(real, name)

    monkeypatch.setattr(_lib, "_lib", Stub())


def _sparse(seed=0, n=30, C=6):
    d = np.random.default_rng(seed).normal(size=(n, C))
    d[d < 0] = 0.0
    return d, sp.csr_matrix(d)


def test_run_edges_and_run_topk_routes(monkeypatch):
    calls = []
    _stub(monkeypatch, calls)
    dense, sparse = _sparse()
    for run, base in ((lambda x, **kw: ik.run_edges(x, (), min_abs_cor=0.5, **kw), "icikt_all_pairs_edges"),
                      (lambda x, **kw: ik.run_topk(x, (), k=3, **kw), "icikt_all_pairs_topk")):
        run(dense, devices=[0, 1, 0])
        assert calls[-1] == dict(name=base + "_multi", C=6, devices=[0, 1, 0])
        run(sparse, devices=(2,))
        assert calls[-1] == dict(name=base + "_multi_csc", C=6, devices=[2])
        run(dense, devices=range(4))
        assert calls[-1]["devices"] == [0, 1, 2, 3]
        run(dense)
        assert calls[-1] == dict(name=base, C=6)
        run(sparse)
        assert calls[-1] == dict(name=base + "_csc", C=6)


def test_ici_kendalltau_topk_n_gpus(monkeypatch):
    calls = []
    _stub(monkeypatch, calls)
    dense, sparse = _sparse(1)
    names = list("abcdef")
    ik.ici_kendalltau_topk(dense, 2, colnames=names, n_gpus=3)
    assert calls[-1] == dict(name="icikt_all_pairs_topk_multi", C=6, devices=[0, 1, 2])
    ik.ici_kendalltau_topk(sparse, 2, colnames=names, n_gpus=2)
    assert calls[-1] == dict(name="icikt_all_pairs_topk_multi_csc", C=6, devices=[0, 1])
    ik.ici_kendalltau_topk(dense, 2, colnames=names)
    assert calls[-1] == dict(name="icikt_all_pairs_topk", C=6)
    ik.ici_kendalltau_topk(dense, 2, colnames=names, n_gpus=1, device=3)
    assert calls[-1] == dict(name="icikt_all_pairs_topk", C=6)


def test_filtered_ici_kendalltau_stays_on_one_gpu(monkeypatch):
    calls = []
    _stub(monkeypatch, calls)
    dense, _ = _sparse(2)
    with pytest.raises(ValueError, match="n_gpus must be 1"):
        ik.ici_kendalltau(dense, colnames=list("abcdef"), return_matrix=False, min_abs_cor=0.3, n_gpus=2)
    assert calls == []
