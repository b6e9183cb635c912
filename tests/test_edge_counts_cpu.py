"""The edge-count calls (icikt_all_pairs_count_edges, icikt_cross_count_edges and their _multi twins) without a GPU:
the ABI, every refusal that comes before any device is touched, the missing device, and the argument checks of the
Python layers."""
import ctypes
import os
import subprocess

import numpy as np
import pytest
import scipy.sparse as sp

import icikendalltau_b200 as ik
from icikendalltau_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAMES = ("icikt_all_pairs_count_edges", "icikt_all_pairs_count_edges_multi", "icikt_cross_count_edges",
         "icikt_cross_count_edges_multi")


def _has_gpu():
    return _lib.load().icikt_device_count() > 0


def _x(n=30, C=6, seed=0):
    return np.asfortranarray(np.random.default_rng(seed).normal(size=(n, C)))


def test_declared_exported_and_bound():
    hdr = open(os.path.join(ROOT, "include", "icikt_b200.h")).read()
    L = ctypes.CDLL(_lib.LIB_PATH)
    for name in NAMES:
        assert name + "(" in hdr, name
        assert hasattr(L, name) and name in _lib.EXPORTS, name
    assert _lib.load().icikt_abi_version() == 1


def test_filters_max_matches_header(tmp_path):
    src = tmp_path / "fmax.c"
    src.write_text('#include <stdio.h>\n#include "icikt_b200.h"\n'
                   'int main(void) { printf("%d %d\\n", ICIKT_COUNT_FILTERS_MAX, ICIKT_NSTATUS); return 0; }\n')
    exe = tmp_path / "fmax"
    subprocess.check_call(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    assert [int(v) for v in subprocess.check_output([str(exe)]).split()] == [_lib.COUNT_FILTERS_MAX, _lib.NSTATUS]
    assert _lib.COUNT_FILTERS_MAX == 64


def _code(fn, *a, **kw):
    with pytest.raises(ik.IciktError) as e:
        fn(*a, **kw)
    return e.value.code


REFUSED_OPTS = [dict(perspective="complete"), dict(kernel=_lib.KERNEL_NAIVE), dict(want_counts=True),
                dict(pair_lo=1, pair_hi=3), dict(pair_hi=3)]


@pytest.mark.parametrize("devices", [None, [0], [0, 0]])
def test_refusals_before_any_device(devices):
    x, y = _x(), _x(C=4, seed=1)
    for run, args in ((ik.run_count_edges, (x,)), (ik.run_cross_count_edges, (x, y))):
        def code(filters=((0.5, None),), **kw):
            return _code(run, *args, (), filters, devices=devices, **kw)
        assert code(filters=()) == _lib.ERR_BAD_ARG                       # T = 0
        assert code(filters=[(0.1, None)] * 65) == _lib.ERR_BAD_ARG       # T = 65
        for kw in REFUSED_OPTS:
            assert code(**kw) == _lib.ERR_BAD_ARG, kw
    assert _code(ik.run_cross_count_edges, x, y, (), ((0.5, None),), devices=devices,
                 include_diag=True) == _lib.ERR_BAD_ARG


def _raw_call(multi=False, cross=False, filters=None, T=1, n_pass=True, n_devices=1, opts=None, x=None):
    """the C entry point with hand-made filters (scale_max, max_edges, reserved) and NULL outputs"""
    L = _lib.load()
    x = _x() if x is None else x
    xi, n, C, keep = _lib._input(x)
    yi, _, Cy, keep_y = _lib._input(_x(C=3, seed=2))
    if filters is None:
        filters = [_lib.EdgeFilter(0.5, float("nan"), 0, 0, 0)]
    arr = (_lib.EdgeFilter * max(len(filters), 1))(*filters)
    np_ = np.zeros(max(T, 1), dtype=np.int64)
    o = opts or _lib.make_opts()
    dev = np.zeros(max(n_devices, 1), dtype=np.int32)
    lead = [ctypes.byref(xi)] + ([ctypes.byref(yi)] if cross else []) + [n, None, 0, ctypes.byref(o)]
    if multi:
        lead += [dev.ctypes.data, n_devices]
    name = ("icikt_cross_count_edges" if cross else "icikt_all_pairs_count_edges") + ("_multi" if multi else "")
    deg = [None, None] if cross else [None]
    return getattr(L, name)(*lead, arr, T, np_.ctypes.data if n_pass else None, *deg, None, None, None)


@pytest.mark.parametrize("multi", [False, True])
@pytest.mark.parametrize("cross", [False, True])
def test_filter_refusals_in_c(multi, cross):
    nan = float("nan")
    bad = [_lib.EdgeFilter(0.5, nan, 1, 0, 0),   # scale_max
           _lib.EdgeFilter(0.5, nan, 0, 0, 10),  # max_edges
           _lib.EdgeFilter(0.5, nan, 0, 1, 0)]   # reserved
    for f in bad:
        assert _raw_call(multi, cross, [_lib.EdgeFilter(0.1, nan, 0, 0, 0), f], T=2) == _lib.ERR_BAD_ARG
    assert _raw_call(multi, cross, n_pass=False) == _lib.ERR_BAD_ARG
    assert _raw_call(multi, cross, T=0) == _lib.ERR_BAD_ARG
    assert _raw_call(multi, cross, T=65, filters=[_lib.EdgeFilter(0.1, nan, 0, 0, 0)] * 65) == _lib.ERR_BAD_ARG
    L = _lib.load()
    xi, n, C, keep = _lib._input(_x())
    np_ = np.zeros(1, dtype=np.int64)
    o = _lib.make_opts()
    assert L.icikt_all_pairs_count_edges(ctypes.byref(xi), n, None, 0, ctypes.byref(o), None, 1, np_.ctypes.data,
                                         None, None, None, None) == _lib.ERR_BAD_ARG  # NULL filters
    if multi:
        assert _raw_call(True, cross, n_devices=0) == _lib.ERR_BAD_ARG
        assert _raw_call(True, cross, n_devices=17) == _lib.ERR_BAD_ARG
    for kw in REFUSED_OPTS:
        assert _raw_call(multi, cross, opts=_lib.make_opts(**kw)) == _lib.ERR_BAD_ARG, kw


def test_bad_csc_is_refused():
    m = sp.random(30, 5, density=0.5, format="csc", random_state=0)
    m.indices[:2] = m.indices[1::-1]  # rows out of order within column 0
    colptr, rowidx = m.indptr.astype(np.int64), m.indices.astype(np.int32)
    xi = _lib.Input(5, None, 0, colptr.ctypes.data, rowidx.ctypes.data, m.data.ctypes.data)
    arr = (_lib.EdgeFilter * 1)(_lib.EdgeFilter(0.5, float("nan"), 0, 0, 0))
    np_ = np.zeros(1, dtype=np.int64)
    o = _lib.make_opts()
    L = _lib.load()
    assert L.icikt_all_pairs_count_edges(ctypes.byref(xi), 30, None, 0, ctypes.byref(o), arr, 1, np_.ctypes.data,
                                         None, None, None, None) == _lib.ERR_BAD_ARG
    assert "matrix x" in L.icikt_last_error().decode()


@pytest.mark.skipif(_has_gpu(), reason="checks the no-GPU behaviour")
def test_well_formed_calls_need_a_device():
    x, y = _x(), _x(C=4, seed=1)
    f = [(0.2, None), (None, 0.05), (None, None)]
    for devices in (None, [0], [0, 1]):
        assert _code(ik.run_count_edges, x, (), f, devices=devices) == _lib.ERR_NO_DEVICE
        assert _code(ik.run_count_edges, sp.csc_matrix(x), (), f, devices=devices,
                     include_diag=True) == _lib.ERR_NO_DEVICE
        assert _code(ik.run_cross_count_edges, x, y, (), f, devices=devices) == _lib.ERR_NO_DEVICE
    assert _raw_call() == _lib.ERR_NO_DEVICE  # every output but n_pass NULL
    names = [f"s{i}" for i in range(6)]
    with pytest.raises(ik.IciktError):
        ik.ici_kendalltau_edge_counts(x, min_abs_cor=[0.1, 0.2], colnames=names)


def test_api_argument_checks():
    x = _x()
    names = [f"s{i}" for i in range(6)]
    with pytest.raises(ValueError, match="at most 64"):
        ik.ici_kendalltau_edge_counts(x, min_abs_cor=np.linspace(0, 1, 9), max_pvalue=np.linspace(0, 1, 8),
                                      colnames=names)
    with pytest.raises(ValueError, match="at most 64"):
        ik.ici_kendalltau_cross_edge_counts(x, x, min_abs_cor=np.linspace(0, 1, 65), xnames=names, ynames=names)
    for bad in ("0.5", True, [0.1, "a"], [[0.1, 0.2]], {"a": 1}):
        with pytest.raises(TypeError):
            ik.ici_kendalltau_edge_counts(x, min_abs_cor=bad, colnames=names)
        with pytest.raises(TypeError):
            ik.ici_kendalltau_cross_edge_counts(x, x, max_pvalue=bad, xnames=names, ynames=names)
    with pytest.raises(ValueError, match="NaN"):
        ik.ici_kendalltau_edge_counts(x, min_abs_cor=float("nan"), colnames=names)
    with pytest.raises(ValueError, match="empty"):
        ik.ici_kendalltau_edge_counts(x, max_pvalue=[], colnames=names)
    with pytest.raises(ValueError, match="Colnames"):
        ik.ici_kendalltau_edge_counts(x, min_abs_cor=0.5)
    with pytest.raises(ValueError, match="No comparisons"):
        ik.ici_kendalltau_edge_counts(x[:, :1], min_abs_cor=0.5, colnames=["a"])
    with pytest.raises(ValueError, match="pair"):
        ik.run_count_edges(x, (), [(0.1, 0.2, 0.3)])


def test_grid_order_and_shape():
    from icikendalltau_b200.api import _count_grid
    f, shape = _count_grid([0.1, 0.2], [1e-3, 1e-2, None])
    assert shape == (2, 3)
    assert f == [(0.1, 1e-3), (0.1, 1e-2), (0.1, None), (0.2, 1e-3), (0.2, 1e-2), (0.2, None)]
    assert _count_grid(0.3, None) == ([(0.3, None)], ())
    assert _count_grid(None, np.array([0.01, 0.05])) == ([(None, 0.01), (None, 0.05)], (2,))
    assert _count_grid(np.float32(0.5), 1) == ([(0.5, 1.0)], ())
    assert _count_grid(np.linspace(0, 1, 8), np.linspace(0, 1, 8))[1] == (8, 8)
