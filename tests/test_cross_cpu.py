"""The cross calls (icikt_cross_pairs, icikt_cross_edges, icikt_cross_topk) without a GPU: the struct layouts, the
argument checks that run before any device is touched, the unit builder of the cross order (compiled for the host from
the header the library uses), and the Python layer with a stand-in for the library."""
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
NAMES = ("icikt_cross_pairs", "icikt_cross_edges", "icikt_cross_topk")


def _has_gpu():
    return _lib.load().icikt_device_count() > 0


# ---------------------------------------------------------------- ABI
def test_struct_sizes_match_header(tmp_path):
    src = tmp_path / "sizes.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "icikt_b200.h"\nint main(void) {\n'
                   '  printf("%zu %zu %zu %zu %zu\\n", sizeof(icikt_input), sizeof(icikt_topk_lists),\n'
                   '         offsetof(icikt_input, colptr), offsetof(icikt_input, values),\n'
                   '         offsetof(icikt_topk_lists, completeness));\n  return 0;\n}\n')
    exe = tmp_path / "sizes"
    subprocess.check_call(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(v) for v in subprocess.check_output([str(exe)]).split()]
    assert got == [ctypes.sizeof(_lib.Input), ctypes.sizeof(_lib.TopkLists), _lib.Input.colptr.offset,
                   _lib.Input.values.offset, _lib.TopkLists.completeness.offset]
    assert set(NAMES) <= set(_lib.EXPORTS)
    assert _lib.load().icikt_abi_version() == 1


# ---------------------------------------------------------------- the unit builder
@pytest.fixture(scope="module")
def host(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("cross") / "libcross_host.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-x", "c++",
                           os.path.join(HERE, "cross_host.cpp"), "-o", out])
    L = ctypes.CDLL(out)
    L.cross_units_host.argtypes = [ctypes.c_longlong] * 6 + [ctypes.c_void_p]
    L.cross_units_host.restype = ctypes.c_longlong
    return L


def _units(L, cx, cy, lo, hi, slots):
    cap = hi - lo + 1
    out = np.zeros((cap, 5), dtype=np.int64)
    m = L.cross_units_host(cx, cy, lo, hi, slots, cap, out.ctypes.data)
    assert m <= cap
    return out[:m]


def _check_cover(U, cx, cy, lo, hi, slots):
    """every pair of [lo, hi) exactly once, at its slot, as (i, Cx + j); units within one x column, in slot order"""
    assert (U[:, 4] == 0).all()
    ulen = max(1, min(16, (hi - lo) // (16 * slots)))
    assert (U[:, 3] >= 1).all() and (U[:, 3] <= ulen).all()
    seen = np.zeros(hi - lo, dtype=np.int64)
    for slot0, col, j0, count, _ in U:
        p = lo + slot0 + np.arange(count)
        assert (p // cy == col).all(), "a unit crosses an x column"
        assert (cx + p % cy == j0 + np.arange(count)).all()
        seen[slot0:slot0 + count] += 1
    assert (seen == 1).all()
    assert (np.diff(U[:, 0]) > 0).all()


@pytest.mark.parametrize("seed", range(6))
def test_cross_units_cover_the_range(host, seed):
    rng = np.random.default_rng(seed)
    cases = [(1, 1, 0, 1, 1), (1, 9, 0, 9, 2), (9, 1, 0, 9, 2), (3, 5, 7, 8, 296), (4, 6, 5, 19, 1), (2, 3, 0, 6, 296)]
    for _ in range(40):
        cx, cy = int(rng.integers(1, 60)), int(rng.integers(1, 300))
        P = cx * cy
        lo = int(rng.integers(0, P))
        hi = int(rng.integers(lo + 1, P + 1))
        cases.append((cx, cy, lo, hi, int(rng.choice([1, 2, 7, 296]))))
    for cx, cy, lo, hi, slots in cases:
        _check_cover(_units(host, cx, cy, lo, hi, slots), cx, cy, lo, hi, slots)


def test_cross_units_windows_of_the_walk(host):
    """the walk cuts [first, last) into windows of W: units restart at every window, mid-row included"""
    cx, cy = 7, 13
    for first, last in ((0, cx * cy), (5, 80)):
        for W in (1, 7, 4096):
            for lo in range(first, last, W):
                hi = min(last, lo + W)
                U = _units(host, cx, cy, lo, hi, 296)
                _check_cover(U, cx, cy, lo, hi, 296)
    assert _units(host, 3, 4, 5, 5, 2).shape[0] == 0
    U = _units(host, 2, 2000, 0, 4000, 1)  # long windows: 16-pair units, cut at the end of a row
    assert U[:, 3].max() == 16 and (U[U[:, 1] == 0][-1, 2] + U[U[:, 1] == 0][-1, 3] == 2 + 2000)


# ---------------------------------------------------------------- argument checks
class Args:
    """valid arguments of one entry point; tests change one thing"""

    def __init__(self, n=20, cx=3, cy=4):
        rng = np.random.default_rng(0)
        self.n = n
        self.x = np.asfortranarray(rng.normal(size=(n, cx)))
        self.y = np.asfortranarray(rng.normal(size=(n, cy)))
        self.xi = _lib.Input(cx, self.x.ctypes.data, n, None, None, None)
        self.yi = _lib.Input(cy, self.y.ctypes.data, n, None, None, None)
        self.opts = _lib.make_opts()
        self.raw = np.full(cx * cy, 7.0)
        self.filter = _lib.EdgeFilter(0.5, float("nan"), 1, 0, 0)
        self.k, self.by = 2, 0
        self.index = np.full((cx, 2), 7, dtype=np.int32)
        self.yindex = np.full((cy, 2), 7, dtype=np.int32)
        self.x_side = _lib.TopkLists(self.index.ctypes.data, None, None, None, None, None, None)
        self.y_side = _lib.TopkLists(self.yindex.ctypes.data, None, None, None, None, None, None)
        self.out = ctypes.c_void_p(7)
        self.use_out = True
        self.use_filter = True
        self.x_ref, self.y_ref = True, True
        self.sides = (True, True)

    def call(self, name):
        L = _lib.load()
        x = ctypes.byref(self.xi) if self.x_ref else None
        y = ctypes.byref(self.yi) if self.y_ref else None
        lead = (x, y, self.n, None, 0, ctypes.byref(self.opts))
        mx = ctypes.c_double()
        if name == "icikt_cross_pairs":
            rc = L.icikt_cross_pairs(*lead, self.raw.ctypes.data if self.raw is not None else None, None, None, None,
                                     None, ctypes.byref(mx), None)
        elif name == "icikt_cross_edges":
            rc = L.icikt_cross_edges(*lead, ctypes.byref(self.filter) if self.use_filter else None,
                                     ctypes.byref(self.out) if self.use_out else None, ctypes.byref(mx), None)
        else:
            rc = L.icikt_cross_topk(*lead, self.k, self.by, 1, ctypes.byref(self.x_side) if self.sides[0] else None,
                                    ctypes.byref(self.y_side) if self.sides[1] else None, ctypes.byref(mx), None)
        return rc, L.icikt_last_error().decode()

    def untouched(self):
        return (self.raw is None or (self.raw == 7.0).all()) and (self.index == 7).all() and (self.yindex == 7).all()


def _bad_csc(a):
    a.yi = _lib.Input(4, None, 0, a.ycsc[0].ctypes.data, a.ycsc[1].ctypes.data, a.ycsc[2].ctypes.data)


def _csc_y(rows):
    def f(a):
        colptr = np.array([0, 2, 4, 5, 6], dtype=np.int64)
        a.ycsc = (colptr, np.array(rows, dtype=np.int32), np.ones(6))
        _bad_csc(a)
    return f


COMMON = {
    "x_null": (lambda a: setattr(a, "x_ref", False), "matrix x"),
    "y_null": (lambda a: setattr(a, "y_ref", False), "matrix y"),
    "both_forms": (lambda a: setattr(a.xi, "colptr", a.x.ctypes.data), "exactly one"),
    "neither_form": (lambda a: setattr(a.yi, "data", None), "exactly one"),
    "x_c_zero": (lambda a: setattr(a.xi, "C", 0), "C must be"),
    "y_c_negative": (lambda a: setattr(a.yi, "C", -1), "C must be"),
    "n_zero": (lambda a: setattr(a, "n", 0), "n must be"),
    "ld_below_n": (lambda a: setattr(a.yi, "ld", 19), "ld must be"),
    "too_many_columns": (lambda a: (setattr(a.xi, "C", 2 ** 31 - 10), setattr(a.yi, "C", 10)), "INT32_MAX"),
    "csc_unsorted": (_csc_y([0, 5, 3, 2, 1, 9]), "matrix y: CSC input: rows of column 1"),
    "csc_row_out_of_range": (_csc_y([0, 5, 2, 3, 25, 9]), "matrix y: CSC input: row 25 of column 2"),
    "include_diag": (lambda a: setattr(a.opts, "include_diag", 1), "include_diag"),
    "complete": (lambda a: setattr(a.opts, "perspective", 2), "perspective"),
    "naive": (lambda a: setattr(a.opts, "kernel", _lib.KERNEL_NAIVE), "tiled kernel"),
    "want_counts": (lambda a: setattr(a.opts, "want_counts", 1), "want_counts"),
}
PAIRS_ONLY = {
    "raw_null": (lambda a: setattr(a, "raw", None), "raw is NULL"),
    "pair_hi_above": (lambda a: setattr(a.opts, "pair_hi", 13), "pair_lo/pair_hi"),
    "pair_lo_above_hi": (lambda a: (setattr(a.opts, "pair_lo", 5), setattr(a.opts, "pair_hi", 4)), "pair_lo/pair_hi"),
    "pair_lo_negative": (lambda a: (setattr(a.opts, "pair_lo", -1), setattr(a.opts, "pair_hi", 4)), "pair_lo/pair_hi"),
    "pair_lo_alone": (lambda a: setattr(a.opts, "pair_lo", 3), "pair_lo/pair_hi"),
}
WHOLE = {
    "pair_lo": (lambda a: (setattr(a.opts, "pair_lo", 1), setattr(a.opts, "pair_hi", 5)), "pair_lo"),
    "pair_hi": (lambda a: setattr(a.opts, "pair_hi", 5), "pair_lo"),
}
EDGES_ONLY = {
    "null_filter": (lambda a: setattr(a, "use_filter", False), "filter is NULL"),
    "null_out": (lambda a: setattr(a, "use_out", False), "out is NULL"),
    "max_edges_negative": (lambda a: setattr(a.filter, "max_edges", -1), "max_edges"),
}
TOPK_ONLY = {
    "k_zero": (lambda a: setattr(a, "k", 0), "k must be"),
    "k_above_max": (lambda a: setattr(a, "k", 1025), "k must be"),
    "by_two": (lambda a: setattr(a, "by", 2), "by must be"),
    "no_side": (lambda a: setattr(a, "sides", (False, False)), "both NULL"),
    "x_side_without_index": (lambda a: setattr(a.x_side, "index", None), "x_side->index"),
    "y_side_without_index": (lambda a: setattr(a.y_side, "index", None), "y_side->index"),
}
CASES = ([("icikt_cross_pairs", c) for c in sorted({**COMMON, **PAIRS_ONLY})] +
         [("icikt_cross_edges", c) for c in sorted({**COMMON, **WHOLE, **EDGES_ONLY})] +
         [("icikt_cross_topk", c) for c in sorted({**COMMON, **WHOLE, **TOPK_ONLY})])
ALL = {**COMMON, **PAIRS_ONLY, **WHOLE, **EDGES_ONLY, **TOPK_ONLY}


@pytest.mark.parametrize("name,case", CASES)
def test_refused_arguments_before_any_device_work(name, case):
    a = Args()
    change, words = ALL[case]
    change(a)
    rc, msg = a.call(name)
    assert rc == _lib.ERR_BAD_ARG, (rc, msg)
    assert words in msg, msg
    assert a.untouched()
    if name == "icikt_cross_edges" and a.use_out:
        assert a.out.value is None  # *out cleared


@pytest.mark.skipif(_has_gpu(), reason="checks the no-GPU behaviour")
@pytest.mark.parametrize("name", NAMES)
def test_no_device(name):
    a = Args()
    rc, msg = a.call(name)
    assert rc == _lib.ERR_NO_DEVICE, msg
    assert a.untouched()
    a = Args()  # CSC on one side, a slice of the pairs
    a.ycsc = (np.array([0, 1, 2, 3, 4], dtype=np.int64), np.array([1, 2, 3, 4], dtype=np.int32), np.ones(4))
    _bad_csc(a)
    a.sides = (False, True)
    if name == "icikt_cross_pairs":
        a.opts.pair_lo, a.opts.pair_hi = 3, 12
    rc, msg = a.call(name)
    assert rc == _lib.ERR_NO_DEVICE, msg
    with pytest.raises(ik.IciktError) as e:
        _lib.run_cross(np.zeros((10, 2)), sp.random(10, 3, density=0.5, format="csc"))
    assert e.value.code == _lib.ERR_NO_DEVICE


def test_python_refusals_before_the_library():
    with pytest.raises(ValueError, match="same rows"):
        _lib.run_cross(np.zeros((10, 2)), np.zeros((11, 2)))
    with pytest.raises(ValueError, match="side"):
        _lib.run_cross_topk(np.zeros((10, 2)), np.zeros((10, 2)), k=1, side="left")
    with pytest.raises(ValueError, match="by must be"):
        _lib.run_cross_topk(np.zeros((10, 2)), np.zeros((10, 2)), k=1, by="max")


# ---------------------------------------------------------------- Python layer with a stand-in library
def _fake_pairs(cx, cy, lo=0, hi=None):
    hi = cx * cy if hi is None else hi
    p = np.arange(lo, hi)
    raw = np.sin(p * 1.7 + 0.3) * 0.9
    status = np.where(p % cy == 2, 3, 0).astype(np.int32)  # y column 2 degenerate
    raw[status != 0] = np.nan
    return dict(raw=raw, pvalue=np.abs(raw) / 10, taumax=np.full(p.size, 0.95), completeness=np.ones(p.size),
                status=status, max_taumax=0.95, timings={})


def _stub(monkeypatch, calls):
    def run_cross(x, y, global_na=(), **kw):
        calls.append(("pairs", x, y, global_na, kw))
        r = _fake_pairs(x.shape[1], y.shape[1])
        calls.append(r)
        return r

    def run_cross_edges(x, y, global_na=(), min_abs_cor=None, max_pvalue=None, scale_max=True, max_edges=0, **kw):
        calls.append(("edges", x, y, global_na, dict(kw, min_abs_cor=min_abs_cor, max_pvalue=max_pvalue,
                                                       scale_max=scale_max, max_edges=max_edges)))
        cy = y.shape[1]
        f = _fake_pairs(x.shape[1], cy)
        cor = f["raw"] / 0.95 if scale_max else f["raw"]
        with np.errstate(invalid="ignore"):
            sel = (f["status"] == 0) & (np.abs(cor) >= (min_abs_cor or 0))
        p = np.nonzero(sel)[0]
        out = dict(i=(p // cy).astype(np.int32), j=(p % cy).astype(np.int32), cor=cor[sel], max_taumax=0.95)
        out.update((k, f[k][sel]) for k in ("raw", "pvalue", "taumax", "completeness"))
        return out

    def run_cross_topk(x, y, global_na=(), k=10, by="abs", scale_max=True, side="both", **kw):
        calls.append(("topk", x, y, global_na, dict(kw, k=k, by=by, scale_max=scale_max, side=side)))
        out = dict(max_taumax=0.95, timings={})
        for s, C, other in (("x", x.shape[1], y.shape[1]), ("y", y.shape[1], x.shape[1])):
            if side in (s, "both"):
                idx = np.full((C, k), -1, dtype=np.int32)
                m = min(k, other)
                idx[:, :m] = np.arange(m)[::-1]
                d = dict(index=idx, n_neighbors=np.full(C, m, dtype=np.int32))
                d.update((f, np.where(idx >= 0, 0.5, np.nan)) for f in _lib.EDGE_NAMES)
                out[s + "_side"] = d
        return out

    for f in (run_cross, run_cross_edges, run_cross_topk):
        monkeypatch.setattr(_lib, f.__name__, f)


def _xy(cx=3, cy=5, n=30):
    rng = np.random.default_rng(cx * 7 + cy)
    return rng.normal(size=(n, cx)), rng.normal(size=(n, cy))


def test_python_full_result_reshaped(monkeypatch):
    calls = []
    _stub(monkeypatch, calls)
    x, y = _xy()
    xn, yn = list("abc"), [f"r{c}" for c in range(5)]
    with pytest.warns(RuntimeWarning, match="single unique value") as rec:
        got = ik.ici_kendalltau_cross(x, y, xnames=xn, ynames=yn, perspective="local", alternative="less",
                                      continuity=True, device=2)
    assert len(rec) == 1  # one warning per class
    kind, _, _, gna, kw = calls[-2]
    assert kind == "pairs" and kw == dict(perspective="local", alternative="less", continuity=True, device=2)
    assert np.isnan(gna[0]) and gna[1:] == [np.inf, 0.0]
    want = _fake_pairs(3, 5)
    for k in ("raw", "pvalue", "taumax", "completeness"):
        assert got[k].shape == (3, 5) and np.array_equal(got[k].ravel(), want[k], equal_nan=True)
    assert np.array_equal(got["cor"], (want["raw"] / 0.95).reshape(3, 5), equal_nan=True)
    assert got["xnames"] == xn and got["ynames"] == yn and got["run_time"] >= 0
    with pytest.warns(RuntimeWarning):
        raw = ik.ici_kendalltau_cross(x, y, xnames=xn, ynames=yn, scale_max=False)
    assert np.array_equal(raw["cor"], raw["raw"], equal_nan=True)
    for k in ("raw", "pvalue", "taumax", "completeness"):  # views of the library's result, not copies
        assert np.shares_memory(raw[k], calls[-1][k])


def test_python_long_table_and_filter(monkeypatch):
    calls = []
    _stub(monkeypatch, calls)
    x, y = _xy()
    xn, yn = list("abc"), list("vwxyz")
    with pytest.warns(RuntimeWarning):
        tab = ik.ici_kendalltau_cross(x, y, xnames=xn, ynames=yn, return_matrix=False)["cor"]
    assert list(tab["s1"]) == [a for a in xn for _ in yn] and list(tab["s2"]) == yn * 3
    assert np.array_equal(tab["raw"], _fake_pairs(3, 5)["raw"], equal_nan=True)
    got = ik.ici_kendalltau_cross(x, y, xnames=xn, ynames=yn, return_matrix=False, min_abs_cor=0.5, max_edges=9)
    kind, _, _, _, kw = calls[-1]
    assert kind == "edges" and kw["min_abs_cor"] == 0.5 and kw["max_edges"] == 9 and kw["scale_max"] is True
    t = got["cor"]
    assert (np.abs(t["cor"]) >= 0.5).all() and set(t["s1"]) <= set(xn) and set(t["s2"]) <= set(yn) - {"x"}
    n_calls = len(calls)
    for kw, words in ((dict(min_abs_cor=0.5), "return_matrix=False"), (dict(return_matrix=False, max_edges=3), "max_edges"),
                      (dict(n_gpus=2), "one GPU")):
        with pytest.raises(ValueError, match=words):
            ik.ici_kendalltau_cross(x, y, xnames=xn, ynames=yn, **kw)
    with pytest.raises(ValueError, match="Colnames of `y`"):
        ik.ici_kendalltau_cross(x, y, xnames=xn)
    with pytest.raises(ValueError, match="same features"):
        ik.ici_kendalltau_cross(x, y[:-1], xnames=xn, ynames=yn)
    assert len(calls) == n_calls


@pytest.mark.parametrize("side", ["x", "y", "both"])
def test_python_topk_sides_and_names(monkeypatch, side):
    calls = []
    _stub(monkeypatch, calls)
    x, y = _xy(2, 6)
    xn, yn = ["q0", "q1"], [f"ref{c}" for c in range(6)]
    got = ik.ici_kendalltau_cross_topk(x, y, np.int64(4), by="signed", side=side, xnames=xn, ynames=yn,
                                       scale_max=False, device=1)
    kind, _, _, _, kw = calls[-1]
    assert kind == "topk" and (kw["k"], kw["by"], kw["side"], kw["scale_max"], kw["device"]) == (4, "signed", side, False, 1)
    assert set(got) == {"x": {"x"}, "y": {"y"}, "both": {"x", "y"}}[side]
    if "x" in got:
        assert got["x"]["neighbors"].shape == (2, 4) and got["x"]["names"] == xn
        assert list(got["x"]["neighbors"][0]) == ["ref3", "ref2", "ref1", "ref0"]
    if "y" in got:
        assert got["y"]["neighbors"].shape == (6, 4) and got["y"]["names"] == yn
        assert list(got["y"]["neighbors"][0]) == ["q1", "q0", None, None]  # k > Cx pads
        assert got["y"]["n_neighbors"][0] == 2
    for bad in (dict(k=0), dict(k=1025), dict(k=2.0), dict(by="max"), dict(side="left"), dict(n_gpus=4)):
        args = dict(k=3)
        args.update(bad)
        with pytest.raises(ValueError):
            ik.ici_kendalltau_cross_topk(x, y, args.pop("k"), xnames=xn, ynames=yn, **args)


def test_python_sparse_and_data_frame_input(monkeypatch):
    calls = []
    _stub(monkeypatch, calls)
    d = np.random.default_rng(2).normal(size=(30, 5))
    d[d < 0] = 0.0
    with pytest.warns(RuntimeWarning):
        ik.ici_kendalltau_cross(sp.csr_matrix(d[:, :2]), d[:, 2:], xnames=list("ab"), ynames=list("cde"))
    _, x, y, _, _ = calls[-2]
    assert sp.issparse(x) and x.format == "csc" and isinstance(y, np.ndarray)  # not densified
    pd = pytest.importorskip("pandas")
    got = ik.ici_kendalltau_cross_topk(pd.DataFrame(d[:, :2], columns=["a", "b"]),
                                       pd.DataFrame(d[:, 2:], columns=["c", "d", "e"]), 2)
    assert got["x"]["names"] == ["a", "b"] and set(got["x"]["neighbors"].ravel()) <= {"c", "d", "e"}


def test_existing_calls_unchanged():
    with pytest.raises(ValueError):
        ik.kt_fast(np.zeros((5, 2)), np.zeros((5, 2)))
