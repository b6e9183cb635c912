"""The top-k all-pairs call (icikt_all_pairs_topk) without a GPU: the header constants, the argument checks that run
before any device is touched, the ranking (compiled for the host from the header the selection kernels use), and
the Python layer with a stand-in for the library."""
import ctypes
import os
import subprocess

import numpy as np
import pytest
import scipy.sparse as sp

import icikendalltau_b200 as ik
from icikendalltau_b200 import _lib

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
NAN = float("nan")
NAMES = ("icikt_all_pairs_topk", "icikt_all_pairs_topk_csc")


def _has_gpu():
    return _lib.load().icikt_device_count() > 0


@pytest.fixture(scope="module")
def host(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("topk") / "libtopk_host.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-x", "c++",
                           os.path.join(HERE, "topk_host.cpp"), "-o", out])
    L = ctypes.CDLL(out)
    vp = ctypes.c_void_p
    L.topk_keys_host.argtypes = [ctypes.c_longlong, vp, ctypes.c_int, vp]
    L.topk_keys_host.restype = None
    L.topk_sort_host.argtypes = [ctypes.c_longlong, vp, vp, ctypes.c_int, vp]
    L.topk_sort_host.restype = None
    return L


# ---------------------------------------------------------------- ABI

def test_header_constants(tmp_path):
    src = tmp_path / "consts.c"
    src.write_text('#include <stdio.h>\n#include "icikt_b200.h"\nint main(void) {\n'
                   '  printf("%d %d %d %d\\n", ICIKT_TOPK_ABS, ICIKT_TOPK_SIGNED, ICIKT_TOPK_MAX, ICIKT_ABI_VERSION);\n'
                   '  return 0;\n}\n')
    exe = tmp_path / "consts"
    subprocess.check_call(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(v) for v in subprocess.check_output([str(exe)]).split()]
    assert got == [_lib.TOPK_BY["abs"], _lib.TOPK_BY["signed"], _lib.TOPK_MAX, 1]
    assert _lib.load().icikt_abi_version() == 1


def _call(name, opts=None, k=4, by=0, index=True, n=20, C=5):
    """one entry point with otherwise valid arguments: (return code, icikt_last_error(), index array)"""
    L = _lib.load()
    o = opts if opts is not None else _lib.make_opts()
    keep = []
    if name == "icikt_all_pairs_topk":
        x = np.asfortranarray(np.random.default_rng(0).normal(size=(n, C)))
        keep.append(x)
        lead = (x.ctypes.data, n, C, n)
    else:
        a = _lib.CSC(sp.random(n, C, density=0.5, format="csc", random_state=1))
        keep.append(a)
        lead = a.args()
    idx = np.full((C, max(k, 1)), 7, dtype=np.int32)
    mx = ctypes.c_double()
    rc = getattr(L, name)(*lead, None, 0, ctypes.byref(o), k, by, 1, idx.ctypes.data if index else None, None,
                          None, None, None, None, None, ctypes.byref(mx), None)
    return rc, L.icikt_last_error().decode(), idx


@pytest.mark.skipif(_has_gpu(), reason="checks the no-GPU behaviour")
@pytest.mark.parametrize("name", NAMES)
def test_no_device(name):
    rc, msg, idx = _call(name)
    assert rc == _lib.ERR_NO_DEVICE, msg
    assert (idx == 7).all()  # nothing written
    with pytest.raises(ik.IciktError) as e:
        _lib.run_topk(np.zeros((10, 3)), k=2)
    assert e.value.code == _lib.ERR_NO_DEVICE


REFUSED = {
    "k_zero": ({}, dict(k=0), "k must be"),
    "k_negative": ({}, dict(k=-3), "k must be"),
    "k_above_max": ({}, dict(k=1025), "k must be"),
    "by_two": ({}, dict(by=2), "by must be"),
    "by_negative": ({}, dict(by=-1), "by must be"),
    "null_index": ({}, dict(index=False), "index is NULL"),
    "include_diag": (dict(include_diag=True), {}, "include_diag"),
    "pair_lo": (dict(pair_lo=1, pair_hi=5), {}, "pair_lo"),
    "pair_hi": (dict(pair_hi=5), {}, "pair_lo"),
    "complete": (dict(perspective="complete"), {}, "perspective"),
    "naive": (dict(kernel=_lib.KERNEL_NAIVE), {}, "tiled kernel"),
    "want_counts": (dict(want_counts=True), {}, "want_counts"),
}


@pytest.mark.parametrize("case", sorted(REFUSED))
@pytest.mark.parametrize("name", NAMES)
def test_refused_arguments_before_any_device_work(name, case):
    okw, ckw, words = REFUSED[case]
    rc, msg, idx = _call(name, opts=_lib.make_opts(**okw), **ckw)
    assert rc == _lib.ERR_BAD_ARG, (rc, msg)
    assert words in msg, msg
    assert (idx == 7).all()


def test_run_topk_refuses_k_through_the_library():
    for k in (0, 1025, 2 ** 32 + 3):
        with pytest.raises(ik.IciktError) as e:
            _lib.run_topk(np.zeros((10, 3)), k=k)
        assert e.value.code == _lib.ERR_BAD_ARG
    with pytest.raises(ValueError, match="by must be"):
        _lib.run_topk(np.zeros((10, 3)), k=2, by="max")


# ---------------------------------------------------------------- the ranking

def _host_order(L, raw, partner, by):
    raw = np.ascontiguousarray(raw, dtype=np.float64)
    partner = np.ascontiguousarray(partner, dtype=np.int32)
    order = np.empty(raw.size, dtype=np.int64)
    L.topk_sort_host(raw.size, raw.ctypes.data, partner.ctypes.data, by, order.ctypes.data)
    return order


def _numpy_order(raw, partner, by):
    return np.lexsort((partner, -np.abs(raw) if by == 0 else -raw))


def _adversarial():
    tiny = np.array([5e-324, 1e-323, 2.2250738585072014e-308 / 3, 2.2250738585072014e-308,
                     np.nextafter(2.2250738585072014e-308, 0)])
    base = np.concatenate([[0.0, -0.0, 1.0, -1.0, 0.5, -0.5, np.nextafter(1.0, 0), -np.nextafter(1.0, 0),
                            np.inf, -np.inf, 1e308, -1e308], tiny, -tiny])
    raw = np.repeat(base, 7)  # equal values with different partners
    return raw


@pytest.mark.parametrize("by", [0, 1])
def test_host_sort_equals_lexsort(host, by):
    rng = np.random.default_rng(11 + by)
    m = 1_000_000
    raw = rng.uniform(-1, 1, size=m)
    raw[: m // 5] = np.round(raw[: m // 5] * 50) / 50     # many equal values
    raw[m // 5: m // 5 + 1000] = rng.choice([0.0, -0.0], size=1000)
    raw = np.concatenate([raw, _adversarial()])
    partner = rng.permutation(raw.size).astype(np.int32)
    got = _host_order(host, raw, partner, by)
    assert np.array_equal(got, _numpy_order(raw, partner, by))


def test_keys(host):
    raw = np.array([0.0, -0.0, 5e-324, -5e-324, 1.0, -1.0, 0.25, -0.25])
    for by in (0, 1):
        key = np.empty(raw.size, dtype=np.uint64)
        host.topk_keys_host(raw.size, raw.ctypes.data, by, key.ctypes.data)
        assert key[0] == key[1]  # -0.0 ranks as +0.0
        if by == 0:
            assert key[2] == key[3] and key[4] == key[5] and key[4] > key[6] > key[2] > key[0]
        else:
            assert key[4] > key[6] > key[2] > key[0] > key[3] > key[7] > key[5]


# ---------------------------------------------------------------- Python layer

def _fake_topk(C, k, by, scale_max):
    """what run_topk returns for a made-up pair result of C columns (column 2 degenerate)"""
    rng = np.random.default_rng(C)
    iu = np.triu_indices(C, 1)
    raw = rng.uniform(-0.9, 0.9, size=iu[0].size)
    ok = (iu[0] != 2) & (iu[1] != 2)
    M = 0.93
    out = dict(index=np.full((C, k), -1, dtype=np.int32), n_neighbors=np.zeros(C, dtype=np.int32),
               max_taumax=M, timings={})
    out.update((name, np.full((C, k), np.nan)) for name in _lib.EDGE_NAMES)
    for c in range(C):
        sel = ok & ((iu[0] == c) | (iu[1] == c))
        d = np.where(iu[0][sel] == c, iu[1][sel], iu[0][sel])
        r = raw[sel]
        o = np.lexsort((d, -np.abs(r) if by == "abs" else -r))[:k]
        m = o.size
        out["index"][c, :m] = d[o]
        out["raw"][c, :m] = r[o]
        out["cor"][c, :m] = r[o] / M if scale_max else r[o]
        out["pvalue"][c, :m] = 0.01
        out["taumax"][c, :m] = M
        out["completeness"][c, :m] = 1.0
        out["n_neighbors"][c] = m
    return out


def _stub(monkeypatch, calls):
    def run_topk(data, global_na=(), k=10, by="abs", scale_max=True, **kw):
        calls.append(dict(data=data, global_na=global_na, k=k, by=by, scale_max=scale_max, **kw))
        return _fake_topk(data.shape[1], k, by, scale_max)
    monkeypatch.setattr(_lib, "run_topk", run_topk)


def test_python_value_errors(monkeypatch):
    calls = []
    _stub(monkeypatch, calls)
    m = np.random.default_rng(0).normal(size=(20, 6))
    names = list("abcdef")
    for k in (0, -1, 1025, 2.5, True, "3", None):
        with pytest.raises(ValueError, match="`k`"):
            ik.ici_kendalltau_topk(m, k, colnames=names)
    for by in ("max", 0, None):
        with pytest.raises(ValueError, match="`by`"):
            ik.ici_kendalltau_topk(m, 2, by=by, colnames=names)
    with pytest.raises(ValueError, match="Colnames"):
        ik.ici_kendalltau_topk(m, 2)
    with pytest.raises(ValueError, match="entries"):
        ik.ici_kendalltau_topk(m, 2, colnames=names[:5])
    assert calls == []


@pytest.mark.parametrize("by", ["abs", "signed"])
@pytest.mark.parametrize("k", [1, 3, 8, 12])
def test_python_shapes_names_and_padding(monkeypatch, by, k):
    calls = []
    _stub(monkeypatch, calls)
    C = 9
    m = np.random.default_rng(1).normal(size=(30, C))
    names = [f"s{c}" for c in range(C)]
    got = ik.ici_kendalltau_topk(m, np.int64(k), by=by, colnames=names, perspective="local", scale_max=False,
                                 alternative="less", continuity=True, device=3)
    call = calls[-1]
    assert call["k"] == k and call["by"] == by and call["scale_max"] is False
    assert (call["perspective"], call["alternative"], call["continuity"], call["device"]) == ("local", "less", True, 3)
    assert np.isnan(call["global_na"][0]) and call["global_na"][1:] == [np.inf, 0.0]
    want = _fake_topk(C, k, by, False)
    for key in ("index", "n_neighbors") + _lib.EDGE_NAMES:
        assert got[key].shape == want[key].shape
        assert np.array_equal(np.asarray(got[key]).view(np.uint8), np.asarray(want[key]).view(np.uint8)), key
    assert got["neighbors"].shape == (C, k) and got["neighbors"].dtype == object
    for c in range(C):
        for r in range(k):
            d = got["index"][c, r]
            assert got["neighbors"][c, r] == (names[d] if d >= 0 else None)
    assert got["n_neighbors"][2] == 0 and (got["index"][2] == -1).all()
    assert (got["n_neighbors"][[0, 1, 3]] == min(k, C - 2)).all()
    assert got["names"] == names and got["run_time"] >= 0 and got["max_taumax"] == 0.93


def test_python_sparse_and_data_frame_input(monkeypatch):
    calls = []
    _stub(monkeypatch, calls)
    d = np.random.default_rng(2).normal(size=(30, 5))
    d[d < 0] = 0.0
    got = ik.ici_kendalltau_topk(sp.csr_matrix(d), 2, colnames=list("vwxyz"))
    assert sp.issparse(calls[-1]["data"]) and calls[-1]["data"].format == "csc"  # not densified
    assert got["neighbors"].shape == (5, 2)
    pd = pytest.importorskip("pandas")
    ik.ici_kendalltau_topk(pd.DataFrame(d, columns=list("abcde")), 2)
    assert isinstance(calls[-1]["data"], np.ndarray) and calls[-1]["data"].dtype == np.float64
    # tuples as names stay whole in the object array
    got = ik.ici_kendalltau_topk(d, 1, colnames=[(c, c + 1) for c in range(5)])
    assert all(isinstance(v, tuple) for v in got["neighbors"][:, 0] if v is not None)
