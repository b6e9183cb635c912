"""Adjusted p-values without a GPU: the NumPy restatement of R's p.adjust (oracle/p_adjust.py) against SciPy and
hand-worked vectors, the per-rank arithmetic of icikt_padj.cuh compiled with g++ against it bit for bit, BY's long
double sum, the ABI of the _padj calls, their refusals before any device work, and the Python argument errors."""
import ctypes
import os
import subprocess

import numpy as np
import pytest
import scipy.stats

from icikendalltau_b200 import _lib, api
from oracle.p_adjust import METHODS, by_q, p_adjust

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
NAN = float("nan")


def _has_gpu():
    try:
        return _lib.load().icikt_device_count() > 0
    except Exception:
        return False


@pytest.fixture(scope="module")
def host(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("padj") / "libpadj_host.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-x", "c++",
                           os.path.join(HERE, "padj_host.cpp"), "-o", out])
    L = ctypes.CDLL(out)
    L.padj_sorted_host.argtypes = [ctypes.c_int, ctypes.c_longlong, ctypes.c_longlong, ctypes.c_void_p,
                                   ctypes.c_double, ctypes.c_void_p]
    L.padj_sorted_host.restype = None
    L.padj_by_q_host.argtypes = [ctypes.c_longlong]
    L.padj_by_q_host.restype = ctypes.c_double
    L.padj_key_host.argtypes = [ctypes.c_double]
    L.padj_key_host.restype = ctypes.c_ulonglong
    return L


def _bits(a):
    return np.asarray(a, dtype=np.float64).view(np.int64)


# ---- the oracle ------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("method", ["BH", "BY"])
def test_oracle_matches_scipy(method):
    rng = np.random.default_rng(7)
    for m in (2, 10, 1000, 100_003):
        p = rng.random(m) ** 3
        p[rng.random(m) < 0.3] = np.round(p[rng.random(m) < 0.3][0], 2)  # ties
        want = scipy.stats.false_discovery_control(p, method=method.lower())
        np.testing.assert_allclose(p_adjust(p, method), want, rtol=1e-14, atol=0)


def test_oracle_hand_worked():
    p = np.array([0.5, 0.25, 0.125, NAN, 0.25])  # m = 4; sorted 0.125, 0.25, 0.25, 0.5
    b = (4.0 / 3.0) * 0.25
    cases = {
        "bonferroni": [1.0, 1.0, 0.5, NAN, 1.0],
        "holm": [0.75, 0.75, 0.5, NAN, 0.75],  # 4, 3, 2, 1 times: 0.5 0.75 0.5 0.5, running max from rank 1
        "hochberg": [0.5, 0.5, 0.5, NAN, 0.5],  # the same values, running min from rank 4
        "BH": [0.5, b, b, NAN, b],  # 0.5, 0.5, (4/3) 0.25, 0.5, running min from rank 4
    }
    for method, want in cases.items():
        assert np.array_equal(_bits(p_adjust(p, method)), _bits(want)), method
    q = 1 + 1 / 2 + 1 / 3 + 1 / 4
    assert p_adjust(p, "BY")[3] != p_adjust(p, "BY")[3]
    assert p_adjust(p, "BY")[0] == min(1.0, ((q * 4) / 4) * 0.5)
    assert np.array_equal(_bits(p_adjust(p, "fdr")), _bits(p_adjust(p, "BH")))
    # zeros and ones; m = 0, 1, 2
    assert list(p_adjust([0.0, 0.0, 1.0], "BH")) == [0.0, 0.0, 1.0]
    for method in METHODS:
        assert np.isnan(p_adjust([NAN, NAN], method)).all()
        assert np.array_equal(_bits(p_adjust([0.3, NAN], method)), _bits([0.3, NAN]))  # m <= 1: p unchanged
        assert p_adjust(np.array([], dtype=np.float64), method).size == 0
    assert list(p_adjust([0.6, 0.2], "bonferroni")) == [1.0, 0.4]
    for method in ("holm", "hochberg", "BH"):
        assert list(p_adjust([0.6, 0.2], method)) == [0.6, 0.4], method


# ---- icikt_padj.cuh on the host ---------------------------------------------------------------------------------

METHOD_CODE = {"bonferroni": 1, "holm": 2, "hochberg": 3, "BH": 4, "BY": 5}


def _host_adjust(host, p, method):
    """p.adjust through icikt_padj.cuh: sort the non-NaN values, scan, put every value back (any order of ties)"""
    p = np.asarray(p, dtype=np.float64)
    ok = ~np.isnan(p)
    x = p[ok]
    m = x.size
    out = p.copy()
    if m <= 1:
        return out
    o = np.argsort(x, kind="quicksort")  # not stable: ties must not matter
    s = np.ascontiguousarray(x[o])
    v = np.empty(m)
    q = host.padj_by_q_host(m) if method == "BY" else 0.0
    host.padj_sorted_host(METHOD_CODE[method], m, m, s.ctypes.data, q, v.ctypes.data)
    adj = np.empty(m)
    adj[o] = v
    out[ok] = adj
    return out


@pytest.mark.parametrize("method", METHODS)
@pytest.mark.parametrize("seed", range(4))
def test_header_arithmetic_bit_for_bit(host, method, seed):
    rng = np.random.default_rng(seed)
    m = [7, 500, 20_000, 3][seed]
    p = rng.random(m) ** 4
    p[rng.random(m) < 0.5] = rng.choice(p, size=1)[0]  # heavy ties
    p[rng.random(m) < 0.2] = np.round(p[rng.random(m) < 0.2], 3)[:1] if m > 3 else p[0]
    p[rng.random(m) < 0.05] = NAN
    p[:1] = 0.0
    assert np.array_equal(_bits(_host_adjust(host, p, method)), _bits(p_adjust(p, method)))


def test_prefix_is_exact(host):
    """the values of the p-values <= alpha from those alone and m, as the device computes them"""
    rng = np.random.default_rng(3)
    p = np.concatenate([rng.random(3000) ** 6, np.full(200, 0.01)])
    for method in METHODS:
        full = p_adjust(p, method)
        for alpha in (1e-6, 0.01, 0.05, 0.5):
            s = np.sort(p[p <= alpha])
            v = np.empty(s.size)
            if s.size == 0:
                continue
            q = by_q(p.size) if method == "BY" else 0.0
            host.padj_sorted_host(METHOD_CODE[method], p.size, s.size, s.ctypes.data, q, v.ctypes.data)
            got = v[np.searchsorted(s, p[p <= alpha], side="right") - 1]
            want = full[p <= alpha]
            keep = want <= alpha
            assert np.array_equal(_bits(got[keep]), _bits(want[keep])), (method, alpha)
            assert (got[~keep] > alpha).all(), (method, alpha)


def test_key_order(host):
    vals = [0.0, 5e-324, 1e-300, 0.01, 0.5, 1.0]
    keys = [host.padj_key_host(v) for v in vals]
    assert keys == sorted(keys)
    assert host.padj_key_host(-0.0) == host.padj_key_host(0.0)


@pytest.mark.skipif(np.finfo(np.longdouble).nmant != 63, reason="needs the 80-bit x87 long double")
@pytest.mark.parametrize("m", [1, 2, 10, 10 ** 6 + 3, 2 ** 24 + 1])
def test_by_sum_bit_for_bit(host, m):
    assert _bits([host.padj_by_q_host(m)])[0] == _bits([by_q(m)])[0]


# ---- ABI -------------------------------------------------------------------------------------------------------

def test_padj_filter_layout_and_constants(tmp_path):
    src = tmp_path / "layout.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "icikt_b200.h"\nint main(void) {\n'
                   '  printf("%zu %zu %zu %zu %d %d %d %d %d\\n", sizeof(icikt_padj_filter), offsetof(icikt_padj_filter, '
                   'method), offsetof(icikt_padj_filter, reserved), offsetof(icikt_padj_filter, max_padj), '
                   'ICIKT_PADJ_BONFERRONI, ICIKT_PADJ_HOLM, ICIKT_PADJ_HOCHBERG, ICIKT_PADJ_BH, ICIKT_PADJ_BY);\n'
                   '  return 0;\n}\n')
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(v) for v in subprocess.check_output([str(exe)]).split()]
    assert got == [16, 0, 4, 8, 1, 2, 3, 4, 5]
    assert ctypes.sizeof(_lib.PadjFilter) == 16 and _lib.PadjFilter.max_padj.offset == 8
    assert {k: v for k, v in _lib.PADJ.items() if k != "fdr"} == METHOD_CODE and _lib.PADJ["fdr"] == 4
    L = _lib.load()
    for name in ("icikt_p_adjust", "icikt_all_pairs_edges_padj", "icikt_all_pairs_edges_padj_multi",
                 "icikt_cross_edges_padj", "icikt_cross_edges_padj_multi", "icikt_edges_copy_padj",
                 "icikt_edges_n_tests"):
        assert hasattr(L, name) and name in _lib.EXPORTS
    assert L.icikt_abi_version() == 1
    assert L.icikt_edges_n_tests(None) == -1
    assert L.icikt_edges_copy_padj(None, None) == _lib.ERR_BAD_ARG


# ---- refusals before any device work ------------------------------------------------------------------------------

def _all_pairs_call(x=True, n=50, adjust=True, method=4, reserved=0, filt=True, out=True, opts=None, devices=None):
    L = _lib.load()
    data = np.asfortranarray(np.random.default_rng(0).random((50, 6)))
    xi = _lib.Input(6, data.ctypes.data, 50, None, None, None)
    o = opts or _lib.make_opts()
    f = _lib.EdgeFilter(NAN, 0.05, 1, 0, 0)
    a = _lib.PadjFilter(method, reserved, 0.05)
    h = ctypes.c_void_p()
    args = [ctypes.byref(xi) if x else None, n, None, 0, ctypes.byref(o)]
    if devices is not None:
        dev = np.asarray(devices, dtype=np.int32)
        args += [dev.ctypes.data, dev.size]
    args += [ctypes.byref(f) if filt else None, ctypes.byref(a) if adjust else None, ctypes.byref(h) if out else None,
             None, None]
    name = "icikt_all_pairs_edges_padj" + ("_multi" if devices is not None else "")
    return getattr(L, name)(*args)


def _cross_call(adjust=True, method=4, reserved=0, opts=None, devices=None):
    L = _lib.load()
    data = np.asfortranarray(np.random.default_rng(0).random((50, 4)))
    xi = _lib.Input(4, data.ctypes.data, 50, None, None, None)
    o = opts or _lib.make_opts()
    f = _lib.EdgeFilter(NAN, NAN, 1, 0, 0)
    a = _lib.PadjFilter(method, reserved, NAN)
    h = ctypes.c_void_p()
    args = [ctypes.byref(xi), ctypes.byref(xi), 50, None, 0, ctypes.byref(o)]
    if devices is not None:
        dev = np.asarray(devices, dtype=np.int32)
        args += [dev.ctypes.data, dev.size]
    args += [ctypes.byref(f), ctypes.byref(a) if adjust else None, ctypes.byref(h), None, None]
    return getattr(_lib.load(), "icikt_cross_edges_padj" + ("_multi" if devices is not None else ""))(*args)


@pytest.mark.parametrize("devices", [None, [0, 0]])
def test_refusals_before_any_device(devices):
    bad = _lib.ERR_BAD_ARG
    assert _all_pairs_call(adjust=False, devices=devices) == bad
    for method in (0, 6, -1):  # 6 would be Hommel's slot: not offered
        assert _all_pairs_call(method=method, devices=devices) == bad
    assert _all_pairs_call(reserved=1, devices=devices) == bad
    assert _all_pairs_call(x=False, devices=devices) == bad
    assert _all_pairs_call(n=0, devices=devices) == bad
    assert _all_pairs_call(n=51, devices=devices) == bad  # ld < n
    assert _all_pairs_call(filt=False, devices=devices) == bad
    assert _all_pairs_call(out=False, devices=devices) == bad
    assert _all_pairs_call(opts=_lib.make_opts(perspective="complete"), devices=devices) == bad
    assert _all_pairs_call(opts=_lib.make_opts(pair_lo=1, pair_hi=3), devices=devices) == bad
    assert _cross_call(adjust=False, devices=devices) == bad
    assert _cross_call(method=0, devices=devices) == bad
    assert _cross_call(reserved=2, devices=devices) == bad
    assert _cross_call(opts=_lib.make_opts(include_diag=True), devices=devices) == bad
    if devices is not None:
        assert _all_pairs_call(devices=[]) == bad
        assert _all_pairs_call(devices=list(range(17))) == bad
        assert _cross_call(devices=list(range(17))) == bad


def test_p_adjust_refusals():
    L = _lib.load()
    p = np.array([0.1, 0.2])
    out = np.empty(2)
    assert L.icikt_p_adjust(p.ctypes.data, -1, 4, 0, out.ctypes.data, None) == _lib.ERR_BAD_ARG
    assert L.icikt_p_adjust(None, 2, 4, 0, out.ctypes.data, None) == _lib.ERR_BAD_ARG
    assert L.icikt_p_adjust(p.ctypes.data, 2, 4, 0, None, None) == _lib.ERR_BAD_ARG
    assert L.icikt_p_adjust(p.ctypes.data, 2, 6, 0, out.ctypes.data, None) == _lib.ERR_BAD_ARG


@pytest.mark.skipif(_has_gpu(), reason="checks the no-GPU behaviour")
def test_well_formed_calls_need_a_device():
    assert _all_pairs_call() == _lib.ERR_NO_DEVICE
    assert _all_pairs_call(devices=[0, 0]) == _lib.ERR_NO_DEVICE
    assert _cross_call() == _lib.ERR_NO_DEVICE
    assert _cross_call(devices=[0]) == _lib.ERR_NO_DEVICE
    p = np.array([0.1, 0.2])
    assert _lib.load().icikt_p_adjust(p.ctypes.data, 2, 4, 0, p.ctypes.data, None) == _lib.ERR_NO_DEVICE
    with pytest.raises(_lib.IciktError) as e:
        _lib.p_adjust(p, "BH")
    assert e.value.code == _lib.ERR_NO_DEVICE


# ---- Python argument errors ---------------------------------------------------------------------------------------

def test_python_argument_errors(monkeypatch):
    x = np.random.default_rng(1).random((20, 5))
    for bad in ("hommel", "bh", "none", 4):
        with pytest.raises(ValueError, match="p_adjust"):
            _lib.p_adjust([0.1], bad)
        with pytest.raises(ValueError, match="p_adjust"):
            _lib.run_edges(x, p_adjust=bad)
    with pytest.raises(ValueError, match="max_padj"):
        _lib.run_edges(x, max_padj=0.05)
    with pytest.raises(ValueError, match="max_padj"):
        _lib.run_cross_edges(x, x, max_padj=0.05)
    with pytest.raises(ValueError, match="return_matrix=False"):
        api.ici_kendalltau(x, p_adjust="BH")
    with pytest.raises(ValueError, match="return_matrix=False"):
        api.ici_kendalltau_cross(x, x, p_adjust="BY", max_padj=0.1)
    with pytest.raises(ValueError, match="give `p_adjust` too"):
        api.ici_kendalltau(x, return_matrix=False, max_padj=0.1)
    with pytest.raises(ValueError, match="n_gpus must be 1"):
        api.ici_kendalltau(x, return_matrix=False, p_adjust="BH", max_padj=0.1, n_gpus=2)
    with pytest.raises(ValueError, match="hommel is not offered"):
        api.ici_kendalltau(x, return_matrix=False, p_adjust="hommel")


def test_python_routing(monkeypatch):
    """filtered tables over all pairs take the windowed _padj call; the unfiltered table and include_only adjust the
    table's p-values with p_adjust and mask on the host"""
    calls = []
    C = 5
    pi, pj = np.triu_indices(C, 1)
    rng = np.random.default_rng(2)
    P = pi.size
    fake = dict(raw=rng.random(P), pvalue=rng.random(P) ** 3, taumax=np.ones(P), completeness=np.ones(P),
                status=np.zeros(P, dtype=np.int32), max_taumax=1.0, timings={})

    def run_pairs(data, global_na=(), pi=None, pj=None, include_diag=False, **kw):
        calls.append("run_pairs")
        return dict(fake)

    def run_edges(data, global_na=(), min_abs_cor=None, max_pvalue=None, scale_max=True, max_edges=0,
                  include_diag=False, p_adjust=None, max_padj=None, **kw):
        calls.append(("run_edges", p_adjust, max_padj))
        padj = p_adjust_oracle(fake["pvalue"], p_adjust)
        sel = padj <= max_padj
        out = dict(i=pi[sel].astype(np.int32), j=pj[sel].astype(np.int32), cor=fake["raw"][sel], padj=padj[sel],
                   n_tests=P, max_taumax=1.0, timings={})
        out.update((k, fake[k][sel]) for k in ("raw", "pvalue", "taumax", "completeness"))
        return out

    p_adjust_oracle = p_adjust
    monkeypatch.setattr(_lib, "run_pairs", run_pairs)
    monkeypatch.setattr(_lib, "run_edges", run_edges)
    monkeypatch.setattr(_lib, "p_adjust", lambda p, method, device=0: p_adjust_oracle(p, method))
    x = rng.random((30, C))
    names = [f"s{c}" for c in range(C)]
    api.ici_kendalltau(x, return_matrix=False, p_adjust="BH", max_padj=0.5, colnames=names)
    assert calls[-1] == ("run_edges", "BH", 0.5)
    r = api.ici_kendalltau(x, return_matrix=False, p_adjust="holm", colnames=names)
    assert calls[-1] == "run_pairs"
    t = r["cor"]
    want = np.concatenate([p_adjust_oracle(fake["pvalue"], "holm"), np.zeros(C)])  # diag_good rows: padj = 0
    assert np.array_equal(t["padj"], want)
    assert (t["s1"][-C:] == t["s2"][-C:]).all()
