"""The filtered all-pairs call (icikt_all_pairs_edges) without a GPU: the ABI, the argument checks that run before
any device is touched, the prefilter against the running maximum (compiled for the host from the header the
selection kernel uses), and the Python layer with a stand-in for the library."""
import ctypes
import os
import subprocess

import numpy as np
import pytest
import scipy.sparse as sp

import icikendalltau_b200 as ik
from icikendalltau_b200 import _lib, api

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
NAN = float("nan")


def _has_gpu():
    return _lib.load().icikt_device_count() > 0


@pytest.fixture(scope="module")
def host(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("edges") / "libedges_host.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-x", "c++",
                           os.path.join(HERE, "edges_host.cpp"), "-o", out])
    L = ctypes.CDLL(out)
    vp = ctypes.c_void_p
    L.prefilter_host.argtypes = [ctypes.c_longlong, vp, vp, vp, vp]
    L.prefilter_host.restype = None
    L.keep_final_host.argtypes = [ctypes.c_longlong, vp, vp, ctypes.c_int, vp, vp]
    L.keep_final_host.restype = None
    L.keep_window_host.argtypes = [ctypes.c_int, ctypes.c_double, ctypes.c_double, ctypes.c_double, ctypes.c_double,
                                   ctypes.c_int, ctypes.c_double]
    L.keep_window_host.restype = ctypes.c_int
    L.edge_row_size.restype = ctypes.c_longlong
    return L


def _prefilter(L, raw, t, m):
    raw, t, m = (np.ascontiguousarray(np.broadcast_to(v, np.shape(raw)), dtype=np.float64) for v in (raw, t, m))
    keep = np.zeros(raw.size, dtype=np.uint8)
    L.prefilter_host(raw.size, raw.ctypes.data, t.ctypes.data, m.ctypes.data, keep.ctypes.data)
    return keep.astype(bool)


def _final(L, raw, t, M, scale_max=True):
    raw, t, M = (np.ascontiguousarray(np.broadcast_to(v, np.shape(raw)), dtype=np.float64) for v in (raw, t, M))
    keep = np.zeros(raw.size, dtype=np.uint8)
    L.keep_final_host(raw.size, raw.ctypes.data, t.ctypes.data, int(scale_max), M.ctypes.data, keep.ctypes.data)
    return keep.astype(bool)


def _exact(raw, t, M):
    with np.errstate(all="ignore"):
        return np.abs(raw / M) >= t  # the IEEE division of the matrix fill and of ici_kendalltau


# ---------------------------------------------------------------- ABI

def test_edge_filter_layout_matches_header(tmp_path):
    assert ctypes.sizeof(_lib.EdgeFilter) == 32
    offs = [getattr(_lib.EdgeFilter, f).offset for f in ("min_abs_cor", "max_pvalue", "scale_max", "reserved",
                                                         "max_edges")]
    src = tmp_path / "layout.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "icikt_b200.h"\nint main(void) {\n'
                   '  printf("%zu %zu %zu %zu %zu %zu %d\\n", sizeof(icikt_edge_filter), offsetof(icikt_edge_filter, '
                   'min_abs_cor), offsetof(icikt_edge_filter, max_pvalue), offsetof(icikt_edge_filter, scale_max), '
                   'offsetof(icikt_edge_filter, reserved), offsetof(icikt_edge_filter, max_edges), ICIKT_ERR_LIMIT);\n'
                   '  return 0;\n}\n')
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(v) for v in subprocess.check_output([str(exe)]).split()]
    assert got == [32] + offs + [_lib.ERR_LIMIT]
    assert _lib.ERR_LIMIT == -6


def test_edge_row_is_40_bytes(host):
    assert host.edge_row_size() == 40


def _call(name, opts=None, filt=True, out=True, max_edges=0, n=20, C=5):
    """one entry point with otherwise valid arguments: (return code, icikt_last_error(), handle)"""
    L = _lib.load()
    o = opts if opts is not None else _lib.make_opts()
    f = _lib.EdgeFilter(0.5, NAN, 1, 0, max_edges)
    h = ctypes.c_void_p(12345)
    mx = ctypes.c_double()
    keep = []
    if name == "icikt_all_pairs_edges":
        x = np.asfortranarray(np.random.default_rng(0).normal(size=(n, C)))
        keep.append(x)
        lead = (x.ctypes.data, n, C, n)
    else:
        a = _lib.CSC(sp.random(n, C, density=0.5, format="csc", random_state=1))
        keep.append(a)
        lead = a.args()
    rc = getattr(L, name)(*lead, None, 0, ctypes.byref(o), ctypes.byref(f) if filt else None,
                          ctypes.byref(h) if out else None, ctypes.byref(mx), None)
    return rc, L.icikt_last_error().decode(), h


NAMES = ("icikt_all_pairs_edges", "icikt_all_pairs_edges_csc")


@pytest.mark.skipif(_has_gpu(), reason="checks the no-GPU behaviour")
@pytest.mark.parametrize("name", NAMES)
def test_no_device(name):
    rc, msg, h = _call(name)
    assert rc == _lib.ERR_NO_DEVICE, msg
    assert h.value is None  # *out is cleared
    with pytest.raises(ik.IciktError) as e:
        _lib.run_edges(np.zeros((10, 3)), min_abs_cor=0.1)
    assert e.value.code == _lib.ERR_NO_DEVICE


REFUSED = {
    "pair_lo": (dict(pair_lo=1, pair_hi=5), {}, "pair_lo"),
    "pair_hi": (dict(pair_hi=5), {}, "pair_lo"),
    "complete": (dict(perspective="complete"), {}, "perspective"),
    "naive": (dict(kernel=_lib.KERNEL_NAIVE), {}, "tiled kernel"),
    "want_counts": (dict(want_counts=True), {}, "want_counts"),
    "max_edges": ({}, dict(max_edges=-1), "max_edges"),
    "null_filter": ({}, dict(filt=False), "filter is NULL"),
    "null_out": ({}, dict(out=False), "out is NULL"),
}


@pytest.mark.parametrize("case", sorted(REFUSED))
@pytest.mark.parametrize("name", NAMES)
def test_refused_arguments_before_any_device_work(name, case):
    okw, ckw, words = REFUSED[case]
    rc, msg, _ = _call(name, opts=_lib.make_opts(**okw), **ckw)
    assert rc == _lib.ERR_BAD_ARG, (rc, msg)
    assert words in msg, msg


def test_edges_handle_helpers():
    L = _lib.load()
    assert L.icikt_edges_count(None) == 0
    assert L.icikt_edges_copy(None, None, None, None, None, None, None, None) == _lib.ERR_BAD_ARG
    L.icikt_edges_free(None)


# ---------------------------------------------------------------- the prefilter against the running maximum

def test_prefilter_never_drops_an_edge_random(host):
    rng = np.random.default_rng(2024)
    m = 1_000_000
    M = np.exp(rng.uniform(np.log(1e-6), np.log(1.0), size=m))
    M[: m // 4] = 1.0
    frac = np.where(rng.random(m) < 0.3, 1.0, rng.random(m) ** rng.choice([1, 4, 40], size=m))
    m_sofar = M * frac                     # M_sofar = M, a little below, and far below
    t = np.where(rng.random(m) < 0.1, 0.0, rng.uniform(0, 1.05, size=m))
    raw = rng.uniform(-1, 1, size=m) * M
    near = rng.random(m) < 0.5             # half of them within a few ulp of the boundary |raw| = t * M
    raw[near] = np.copysign(t[near] * M[near], raw[near])
    raw[near] = raw[near] + rng.integers(-4, 5, size=int(near.sum())) * np.spacing(raw[near])
    ex = _exact(raw, t, M)
    pre = _prefilter(host, raw, t, m_sofar)
    assert ex.sum() > m // 10
    assert not (ex & ~pre).any(), np.nonzero(ex & ~pre)[0][:5]
    assert np.array_equal(_final(host, raw, t, M), ex)  # the final trim is the exact predicate


def test_prefilter_adversarial_cases(host):
    cases = []
    for M in (1.0, 0.999999, 0.73, 0.5, 3e-3, 1e-300, 2.0 ** -1000, 1e300):
        for frac in (1.0, 1 - 2 ** -52, 0.999, 0.5, 1e-3, 1e-30, 2 ** -1074):
            ms = M * frac
            if ms == 0:
                continue
            for t in (0.0, 5e-324, 2.0 ** -1000, 1e-300, 1e-17, 0.1, 0.3, 0.5, 1.0 / 3, 0.9999999999, 1.0, 1.01,
                      2.0 ** 1000, 1e308, np.inf):
                b = t * M
                for r in (b, np.nextafter(b, 0), np.nextafter(b, np.inf), np.nextafter(np.nextafter(b, 0), 0),
                          5e-324, 2.2250738585072014e-308 / 3, 0.0, M, 1.0):
                    for s in (1.0, -1.0):
                        cases.append((s * r, t, ms, M))
    raw, t, ms, M = (np.array(c, dtype=np.float64) for c in zip(*cases))
    finite = np.isfinite(raw)
    raw, t, ms, M = raw[finite], t[finite], ms[finite], M[finite]
    ex = _exact(raw, t, M)
    pre = _prefilter(host, raw, t, ms)
    bad = np.nonzero(ex & ~pre)[0]
    assert bad.size == 0, [(raw[k], t[k], ms[k], M[k]) for k in bad[:5]]
    assert np.array_equal(_final(host, raw, t, M), ex)
    # t = 0 keeps everything, subnormal raw included
    assert _prefilter(host, np.array([5e-324, -0.0, 0.0]), 0.0, 1.0).all()


def test_prefilter_at_the_final_maximum_is_tight(host):
    """with M_sofar = M the prefilter keeps the edges plus only rows within a relative 2^-49 of the boundary,
    which the final trim removes"""
    rng = np.random.default_rng(7)
    m = 1_000_000
    M = rng.uniform(0.2, 1.0, size=m)
    t = rng.uniform(0.01, 1.0, size=m)
    raw = rng.uniform(-1, 1, size=m) * M
    near = rng.random(m) < 0.5
    raw[near] = np.copysign(t[near] * M[near], raw[near]) * (1 + rng.integers(-40, 41, size=int(near.sum())) * 2.0 ** -53)
    ex = _exact(raw, t, M)
    pre = _prefilter(host, raw, t, M)
    assert not (ex & ~pre).any()
    extra = pre & ~ex
    assert extra.sum() < near.sum() // 4
    assert (np.abs(raw[extra]) >= t[extra] * M[extra] * (1 - 2.0 ** -49)).all()
    assert np.array_equal((pre & _final(host, raw, t, M)), ex)


def test_window_predicate(host):
    kw = host.keep_window_host
    assert kw(0, 0.3, 0.01, NAN, NAN, 1, 1.0) == 1       # no bound: every valid pair
    assert kw(2, 0.3, 0.01, NAN, NAN, 1, 1.0) == 0       # degenerate pairs never
    assert kw(0, 0.3, NAN, 0.0, NAN, 0, 1.0) == 1        # n = 2: NaN p-value kept under min_abs_cor alone
    assert kw(0, 0.3, NAN, NAN, 1.0, 0, 1.0) == 0        # ... and dropped under max_pvalue
    assert kw(0, -0.3, 0.2, 0.3, NAN, 0, 1.0) == 1       # without scale_max the cor test is exact
    assert kw(0, np.nextafter(0.3, 0), 0.2, 0.3, NAN, 0, 1.0) == 0
    assert kw(0, 0.3, 0.2, 0.5, NAN, 1, 0.6) == 1        # 0.3 >= 0.5 * 0.6 (1 - 2^-50)
    assert kw(0, 0.29, 0.2, 0.5, NAN, 1, 0.6) == 0
    assert kw(0, 0.9, 0.2, NAN, 0.1, 1, 1.0) == 0        # p-value bound is exact
    assert kw(0, 0.9, 0.1, NAN, 0.1, 1, 1.0) == 1


# ---------------------------------------------------------------- Python layer

def test_python_value_errors():
    m = np.random.default_rng(0).normal(size=(20, 6))
    names = list("abcdef")
    with pytest.raises(ValueError, match="return_matrix=False"):
        ik.ici_kendalltau(m, colnames=names, min_abs_cor=0.5)
    with pytest.raises(ValueError, match="return_matrix=False"):
        ik.ici_kendalltau(m, colnames=names, max_pvalue=0.05, return_matrix=True)
    with pytest.raises(ValueError, match="n_gpus must be 1"):
        ik.ici_kendalltau(m, colnames=names, min_abs_cor=0.5, return_matrix=False, n_gpus=2)
    with pytest.raises(ValueError, match="max_edges"):
        ik.ici_kendalltau(m, colnames=names, return_matrix=False, max_edges=10)


def _fake_pairs(C, include_diag, seed=0):
    """a per-pair result of C columns in the library's pair order, with degenerate pairs and a NaN p-value"""
    rng = np.random.default_rng(seed)
    iu = np.triu_indices(C, 1)
    pi, pj = iu[0].astype(np.int32), iu[1].astype(np.int32)
    if include_diag:
        d = np.arange(C, dtype=np.int32)
        pi, pj = np.concatenate([pi, d]), np.concatenate([pj, d])
    P = pi.size
    raw = rng.uniform(-0.9, 0.9, size=P)
    pv = rng.uniform(0, 0.2, size=P) ** 2
    tm = rng.uniform(0.5, 0.95, size=P)
    comp = rng.uniform(0.5, 1, size=P)
    status = np.zeros(P, dtype=np.int32)
    status[::7] = 2
    for a in (raw, pv, tm, comp):
        a[status != 0] = np.nan
    pv[3] = np.nan
    return pi, pj, dict(raw=raw, pvalue=pv, taumax=tm, completeness=comp, status=status,
                        max_taumax=float(np.nanmax(tm)), timings={})


def _stub(monkeypatch, calls, C):
    def run_pairs(data, global_na=(), pi=None, pj=None, include_diag=False, **kw):
        api, apj, r = _fake_pairs(C, include_diag or pi is not None)
        if pi is not None:
            code = api.astype(np.int64) * C + apj
            idx = np.array([np.nonzero(code == a * C + b)[0][0] for a, b in zip(pi, pj)])
            r = {k: (v[idx] if isinstance(v, np.ndarray) else v) for k, v in r.items()}
            r["max_taumax"] = float(np.nanmax(r["taumax"]))
        calls.append(("run_pairs", pi is not None))
        return r

    def run_edges(data, global_na=(), min_abs_cor=None, max_pvalue=None, scale_max=True, max_edges=0,
                  include_diag=False, **kw):
        pi, pj, r = _fake_pairs(C, include_diag)
        cor = r["raw"] / r["max_taumax"] if scale_max else r["raw"].copy()
        sel = r["status"] == 0
        if min_abs_cor is not None:
            sel &= np.abs(cor) >= min_abs_cor
        if max_pvalue is not None:
            sel &= r["pvalue"] <= max_pvalue
        calls.append(("run_edges", max_edges))
        out = dict(i=pi[sel], j=pj[sel], cor=cor[sel], max_taumax=r["max_taumax"], timings={})
        out.update((k, r[k][sel]) for k in ("raw", "pvalue", "taumax", "completeness"))
        return out

    monkeypatch.setattr(_lib, "run_pairs", run_pairs)
    monkeypatch.setattr(_lib, "run_edges", run_edges)

    def no_list(*a, **k):
        raise AssertionError("the pair list was built on the host")
    return no_list


def _masked(table, t, a):
    sel = np.ones(len(table["cor"]), dtype=bool)
    if t is not None:
        sel &= np.abs(table["cor"]) >= t
    if a is not None:
        sel &= table["pvalue"] <= a
    return {k: np.asarray(v)[sel] for k, v in table.items()}


@pytest.mark.parametrize("diag_good", [True, False])
@pytest.mark.parametrize("scale_max", [True, False])
@pytest.mark.parametrize("bounds", [(0.3, None), (None, 0.01), (0.2, 1e-3), (0.0, None), (1.01, None)])
def test_filtered_long_table_equals_the_masked_table(monkeypatch, diag_good, scale_max, bounds):
    C = 9
    calls = []
    no_list = _stub(monkeypatch, calls, C)
    m = np.random.default_rng(1).normal(size=(30, C))
    m[:4, 2] = np.nan
    names = [f"s{k}" for k in range(C)]
    t, a = bounds
    kw = dict(colnames=names, return_matrix=False, diag_good=diag_good, scale_max=scale_max)
    with pytest.warns(RuntimeWarning):
        full = ik.ici_kendalltau(m, **kw)["cor"]
    want = _masked(full, t, a)
    monkeypatch.setattr(api, "setup_comparisons", no_list)
    got = ik.ici_kendalltau(m, min_abs_cor=t, max_pvalue=a, max_edges=10 ** 6, **kw)["cor"]
    monkeypatch.undo()
    assert calls[-1] == ("run_edges", 10 ** 6)
    assert set(got) == set(want)
    for k in want:
        if want[k].dtype == object:
            assert list(got[k]) == list(want[k]), k
        else:
            assert np.array_equal(got[k].view(np.int64), want[k].view(np.int64)), k
    # include_only: the pair list exists, the mask runs on the host
    _stub(monkeypatch, calls, C)
    with pytest.warns(RuntimeWarning):
        full = ik.ici_kendalltau(m, include_only=["s1", "s4"], **kw)["cor"]
    want = _masked(full, t, a)
    with pytest.warns(RuntimeWarning):  # the per-pair call reports degenerate pairs as before
        got = ik.ici_kendalltau(m, include_only=["s1", "s4"], min_abs_cor=t, max_pvalue=a, **kw)["cor"]
    assert calls[-1] == ("run_pairs", True)
    for k in want:
        if want[k].dtype == object:
            assert list(got[k]) == list(want[k]), k
        else:
            assert np.array_equal(np.asarray(got[k]).view(np.int64), want[k].view(np.int64)), k


def test_include_only_max_edges(monkeypatch):
    C = 9
    _stub(monkeypatch, [], C)
    m = np.random.default_rng(1).normal(size=(30, C))
    names = [f"s{k}" for k in range(C)]
    with pytest.raises(ik.IciktError) as e, pytest.warns(RuntimeWarning):
        ik.ici_kendalltau(m, colnames=names, include_only=["s1", "s4"], return_matrix=False, min_abs_cor=0.0,
                          max_edges=2)
    assert e.value.code == _lib.ERR_LIMIT
