"""The component calls (icikt_all_pairs_components, icikt_cross_components and their _multi twins) without a GPU: the
ABI, every refusal that comes before any device is touched, the missing device, the API's argument checks, and the
union-find of icikt_components.cuh compiled with g++ -- the host merge of several devices' labels and a sequential run
of the find and hook the tally kernel runs -- against scipy's connected components."""
import ctypes
import os
import subprocess

import numpy as np
import pytest
import scipy.sparse as sp
from scipy.sparse.csgraph import connected_components

import icikendalltau_b200 as ik
from icikendalltau_b200 import _lib

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
NAMES = ("icikt_all_pairs_components", "icikt_all_pairs_components_multi", "icikt_cross_components",
         "icikt_cross_components_multi")


def _has_gpu():
    return _lib.load().icikt_device_count() > 0


def _x(n=30, C=6, seed=0):
    return np.asfortranarray(np.random.default_rng(seed).normal(size=(n, C)))


def _code(fn, *a, **kw):
    with pytest.raises(ik.IciktError) as e:
        fn(*a, **kw)
    return e.value.code


def test_declared_exported_and_bound():
    hdr = open(os.path.join(ROOT, "include", "icikt_b200.h")).read()
    L = ctypes.CDLL(_lib.LIB_PATH)
    for name in NAMES:
        assert name + "(" in hdr, name
        assert hasattr(L, name) and name in _lib.EXPORTS, name


def _raw_call(multi=False, cross=False, filters=None, T=1, n_pass=True, comp=(True, True), n_devices=1, opts=None):
    """the C entry point with hand-made filters and NULL outputs; comp: whether component (all-pairs) or x_component,
    y_component (cross) are given"""
    L = _lib.load()
    xi, n, C, keep = _lib._input(_x())
    yi, _, Cy, keep_y = _lib._input(_x(C=3, seed=2))
    if filters is None:
        filters = [_lib.EdgeFilter(0.5, float("nan"), 0, 0, 0)]
    arr = (_lib.EdgeFilter * max(len(filters), 1))(*filters)
    np_ = np.zeros(max(T, 1), dtype=np.int64)
    xc, yc = np.zeros(C * 64, dtype=np.int32), np.zeros(Cy * 64, dtype=np.int32)
    o = opts or _lib.make_opts()
    dev = np.zeros(max(n_devices, 1), dtype=np.int32)
    lead = [ctypes.byref(xi)] + ([ctypes.byref(yi)] if cross else []) + [n, None, 0, ctypes.byref(o)]
    if multi:
        lead += [dev.ctypes.data, n_devices]
    name = ("icikt_cross_components" if cross else "icikt_all_pairs_components") + ("_multi" if multi else "")
    labels = [xc.ctypes.data if comp[0] else None] + ([yc.ctypes.data if comp[1] else None] if cross else [])
    deg = [None, None] if cross else [None]
    return getattr(L, name)(*lead, arr, T, np_.ctypes.data if n_pass else None, *deg, *labels, None, None, None,
                            None)


REFUSED_OPTS = [dict(perspective="complete"), dict(kernel=_lib.KERNEL_NAIVE), dict(want_counts=True),
                dict(pair_lo=1, pair_hi=3), dict(pair_hi=3)]


@pytest.mark.parametrize("multi", [False, True])
@pytest.mark.parametrize("cross", [False, True])
def test_refusals_in_c(multi, cross):
    nan = float("nan")
    L = _lib.load()
    # the new ones: no label table at all
    assert _raw_call(multi, cross, comp=(False, False)) == _lib.ERR_BAD_ARG
    msg = L.icikt_last_error().decode()
    assert ("both NULL" in msg) if cross else ("component is NULL" in msg), msg
    # the inherited ones, with the count calls' messages
    for f, text in ((_lib.EdgeFilter(0.5, nan, 1, 0, 0), "scale_max"), (_lib.EdgeFilter(0.5, nan, 0, 0, 10), "max_edges"),
                    (_lib.EdgeFilter(0.5, nan, 0, 1, 0), "reserved")):
        assert _raw_call(multi, cross, [_lib.EdgeFilter(0.1, nan, 0, 0, 0), f], T=2) == _lib.ERR_BAD_ARG
        assert text in L.icikt_last_error().decode()
    assert _raw_call(multi, cross, n_pass=False) == _lib.ERR_BAD_ARG
    assert _raw_call(multi, cross, T=0) == _lib.ERR_BAD_ARG
    assert _raw_call(multi, cross, T=65, filters=[_lib.EdgeFilter(0.1, nan, 0, 0, 0)] * 65) == _lib.ERR_BAD_ARG
    if multi:
        assert _raw_call(True, cross, n_devices=0) == _lib.ERR_BAD_ARG
        assert _raw_call(True, cross, n_devices=17) == _lib.ERR_BAD_ARG
    for kw in REFUSED_OPTS:
        assert _raw_call(multi, cross, opts=_lib.make_opts(**kw)) == _lib.ERR_BAD_ARG, kw


@pytest.mark.parametrize("devices", [None, [0], [0, 0]])
def test_python_refusals_before_any_device(devices):
    x, y = _x(), _x(C=4, seed=1)
    for run, args in ((ik.run_count_edges, (x,)), (ik.run_cross_count_edges, (x, y))):
        assert _code(run, *args, (), (), devices=devices, want_components=True) == _lib.ERR_BAD_ARG
        for kw in REFUSED_OPTS:
            assert _code(run, *args, (), ((0.5, None),), devices=devices, want_components=True,
                         **kw) == _lib.ERR_BAD_ARG, kw
    assert _code(ik.run_cross_count_edges, x, y, (), ((0.5, None),), devices=devices, include_diag=True,
                 want_components=True) == _lib.ERR_BAD_ARG


@pytest.mark.skipif(_has_gpu(), reason="checks the no-GPU behaviour")
def test_well_formed_calls_need_a_device():
    x, y = _x(), _x(C=4, seed=1)
    f = [(0.2, None), (None, 0.05)]
    for devices in (None, [0], [0, 1]):
        assert _code(ik.run_count_edges, x, (), f, devices=devices, want_components=True) == _lib.ERR_NO_DEVICE
        assert _code(ik.run_count_edges, sp.csc_matrix(x), (), f, devices=devices, include_diag=True,
                     want_components=True) == _lib.ERR_NO_DEVICE
        assert _code(ik.run_cross_count_edges, x, y, (), f, devices=devices,
                     want_components=True) == _lib.ERR_NO_DEVICE
    assert _raw_call() == _lib.ERR_NO_DEVICE
    assert _raw_call(cross=True, comp=(False, True)) == _lib.ERR_NO_DEVICE  # one side is enough
    assert _raw_call(cross=True, comp=(True, False), multi=True) == _lib.ERR_NO_DEVICE
    names = [f"s{i}" for i in range(6)]
    with pytest.raises(ik.IciktError):
        ik.ici_kendalltau_edge_counts(x, min_abs_cor=[0.1, 0.2], colnames=names, components=True)


def test_api_argument_checks():
    x = _x()
    names = [f"s{i}" for i in range(6)]
    with pytest.raises(ValueError, match="at most 64"):
        ik.ici_kendalltau_edge_counts(x, min_abs_cor=np.linspace(0, 1, 65), colnames=names, components=True)
    with pytest.raises(ValueError, match="at most 64"):
        ik.ici_kendalltau_cross_edge_counts(x, x, min_abs_cor=np.linspace(0, 1, 65), xnames=names, ynames=names,
                                            components=True)
    with pytest.raises(TypeError):
        ik.ici_kendalltau_edge_counts(x, min_abs_cor="0.5", colnames=names, components=True)
    with pytest.raises(ValueError, match="Colnames"):
        ik.ici_kendalltau_edge_counts(x, min_abs_cor=0.5, components=True)
    with pytest.raises(ValueError, match="No comparisons"):
        ik.ici_kendalltau_edge_counts(x[:, :1], min_abs_cor=0.5, colnames=["a"], components=True)


# ---------------------------------------------------------------- the union-find, compiled with g++

@pytest.fixture(scope="module")
def host(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("components") / "libcomponents_host.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-x", "c++",
                           os.path.join(HERE, "components_host.cpp"), "-o", out])
    L = ctypes.CDLL(out)
    vp = ctypes.c_void_p
    L.merge_host.argtypes = [ctypes.c_int, ctypes.c_longlong, ctypes.c_int, vp, vp, vp]
    L.merge_host.restype = None
    L.unite_host.argtypes = [ctypes.c_longlong, ctypes.c_longlong, vp, vp, vp]
    L.unite_host.restype = ctypes.c_longlong
    return L


def reference(V, a, b):
    """(labels as the smallest vertex of each component, number of components) by scipy"""
    g = sp.coo_matrix((np.ones(len(a)), (np.asarray(a), np.asarray(b))), shape=(V, V))
    n, lab = connected_components(g, directed=False)
    first = np.full(n, V, dtype=np.int64)
    np.minimum.at(first, lab, np.arange(V))
    return first[lab].astype(np.int32), n


def unite(host, V, a, b):
    a, b = np.ascontiguousarray(a, dtype=np.int32), np.ascontiguousarray(b, dtype=np.int32)
    lab = np.empty(V, dtype=np.int32)
    hooks = host.unite_host(V, a.size, a.ctypes.data, b.ctypes.data, lab.ctypes.data)
    assert hooks >= 0, "parent[v] <= v broken"
    return lab, hooks


def merge(host, T, V, tables):
    """tables: K arrays of [T][V] labels"""
    lab = np.ascontiguousarray(np.stack(tables), dtype=np.int32)
    out = np.empty((T, V), dtype=np.int32)
    n = np.empty(T, dtype=np.int64)
    host.merge_host(T, V, len(tables), lab.ctypes.data, out.ctypes.data, n.ctypes.data)
    return out, n


def test_sequential_unions_match_scipy(host):
    rng = np.random.default_rng(1)
    for trial in range(2000):
        V = int(rng.integers(1, 60))
        m = int(rng.integers(0, 2 * V + 1))
        a, b = rng.integers(0, V, m), rng.integers(0, V, m)
        lab, hooks = unite(host, V, a, b)
        ref, n = reference(V, a, b)
        assert np.array_equal(lab, ref), trial
        assert V - hooks == n, trial


def test_merge_of_random_device_slices(host):
    """10^4 random graphs, their edges split over 1..16 'devices' whose labels come from the sequential unions"""
    rng = np.random.default_rng(2)
    for trial in range(10000):
        V = int(rng.integers(1, 40))
        T = int(rng.integers(1, 4))
        K = int(rng.integers(1, 17))
        tables = [np.empty((T, V), dtype=np.int32) for _ in range(K)]
        refs = []
        for f in range(T):
            m = int(rng.integers(0, 2 * V + 1))
            a, b = rng.integers(0, V, m), rng.integers(0, V, m)
            dev = rng.integers(0, K, m)
            for k in range(K):
                tables[k][f] = unite(host, V, a[dev == k], b[dev == k])[0]
            refs.append(reference(V, a, b))
        out, n = merge(host, T, V, tables)
        for f in range(T):
            assert np.array_equal(out[f], refs[f][0]), (trial, f)
            assert n[f] == refs[f][1], (trial, f)


def test_chains_against_naive_linking(host):
    """long chains whose edges come in the orders that make naive linking deep or quadratic: descending, ascending,
    alternating ends, and each device holding every K-th link"""
    V = 20000
    v = np.arange(V - 1)
    orders = {"ascending": v, "descending": v[::-1], "ends": np.ravel(np.column_stack([v[: V // 2], v[::-1][: V // 2]]))[: V - 1]}
    for name, o in orders.items():
        lab, hooks = unite(host, V, o, o + 1)
        assert hooks == V - 1 and not lab.any(), name
        lab, hooks = unite(host, V, o + 1, o)  # the larger endpoint first
        assert hooks == V - 1 and not lab.any(), name
    for K in (2, 3, 16):
        tables = [unite(host, V, v[k::K], v[k::K] + 1)[0][None, :] for k in range(K)]
        out, n = merge(host, 1, V, tables)
        assert n[0] == 1 and not out.any(), K
    # two interleaved chains (evens, odds) that only one edge joins, given to another device
    ev, od = np.arange(0, V - 2, 2), np.arange(1, V - 2, 2)
    t0 = unite(host, V, np.concatenate([ev, od]), np.concatenate([ev + 2, od + 2]))[0]
    out, n = merge(host, 1, V, [t0[None, :]])
    assert n[0] == 2 and set(np.unique(out)) == {0, 1}
    t1 = unite(host, V, [V - 1], [V - 2])[0]
    out, n = merge(host, 1, V, [t0[None, :], t1[None, :]])
    assert n[0] == 1 and not out.any()
