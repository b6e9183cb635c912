"""Sparse (CSC) input without a GPU: the host-side checks of the *_csc entry points, and what the Python
layer hands to them (checked with ctypes stand-ins for the library calls)."""
import ctypes

import numpy as np
import pytest
import scipy.sparse as sp

import icikendalltau_b200 as ik
from icikendalltau_b200 import _lib

NAMES = ("icikt_all_pairs_csc", "icikt_all_pairs_multi_csc", "icikt_pair_list_csc", "icikt_matrices_csc",
         "icikt_matrices_multi_csc", "icikt_pairwise_completeness_csc")


def _call(name, colptr, rowidx, values, n, C):
    """one *_csc entry point with otherwise valid arguments: (return code, icikt_last_error())"""
    L = _lib.load()
    colptr = np.ascontiguousarray(colptr, dtype=np.int64)
    rowidx = None if rowidx is None else np.ascontiguousarray(rowidx, dtype=np.int32)
    values = None if values is None else np.ascontiguousarray(values, dtype=np.float64)
    lead = (_lib._ptr(colptr), _lib._ptr(rowidx), _lib._ptr(values), n, C)
    P = C * (C - 1) // 2 + C
    out = np.zeros(5 * P + C * C * 5 + 16)
    o = _lib.make_opts()
    pi = np.zeros(1, dtype=np.int32)
    dev = np.zeros(1, dtype=np.int32)
    hist = np.zeros(_lib.NSTATUS, dtype=np.int64)
    a = out.ctypes.data
    mx, t = ctypes.c_double(), _lib.Timings()
    f = getattr(L, name)
    if name == "icikt_all_pairs_csc":
        rc = f(*lead, None, 0, ctypes.byref(o), a, None, None, None, None, None, ctypes.byref(mx), ctypes.byref(t))
    elif name == "icikt_all_pairs_multi_csc":
        rc = f(*lead, None, 0, ctypes.byref(o), dev.ctypes.data, 1, a, None, None, None, None, None, ctypes.byref(mx),
               ctypes.byref(t))
    elif name == "icikt_pair_list_csc":
        rc = f(*lead, None, 0, pi.ctypes.data, pi.ctypes.data, 1, ctypes.byref(o), a, None, None, None, None, None,
               ctypes.byref(mx), ctypes.byref(t))
    elif name == "icikt_matrices_csc":
        rc = f(*lead, None, 0, None, None, 0, ctypes.byref(o), 1, 1, None, a, None, None, None, None,
               hist.ctypes.data, ctypes.byref(mx), ctypes.byref(t))
    elif name == "icikt_matrices_multi_csc":
        rc = f(*lead, None, 0, ctypes.byref(o), dev.ctypes.data, 1, 1, 1, None, a, None, None, None, None,
               hist.ctypes.data, ctypes.byref(mx), ctypes.byref(t))
    else:
        rc = f(*lead, None, 0, 0, None, None, P, None, None, a)
    return rc, L.icikt_last_error().decode()


# colptr, rowidx, n, C, words the message must contain
BAD = {
    "colptr0": ([1, 2, 3], [0, 1], 4, 2, ["colptr[0]", "not 0"]),
    "decreasing": ([0, 2, 1, 3], [0, 1, 2], 4, 3, ["decreases", "column 1"]),
    "entries_without_arrays": ([0, 1, 2], None, 4, 2, ["colptr[C] = 2", "NULL"]),
    "row_too_large": ([0, 1, 3], [0, 1, 4], 4, 2, ["row 4", "column 1", "[0, 4)"]),
    "row_negative": ([0, 2, 2], [-1, 1], 4, 2, ["row -1", "column 0"]),
    "unsorted": ([0, 1, 4], [2, 3, 1, 2], 4, 2, ["column 1", "not sorted", "3 before 1"]),
    "duplicate": ([0, 3, 3], [0, 2, 2], 4, 2, ["column 0", "repeat row 2"]),
}


@pytest.mark.parametrize("case", sorted(BAD))
@pytest.mark.parametrize("name", NAMES)
def test_csc_checks_run_on_the_host(name, case):
    colptr, rowidx, n, C, words = BAD[case]
    values = None if rowidx is None else np.arange(len(rowidx), dtype=np.float64)
    rc, msg = _call(name, colptr, rowidx, values, n, C)
    assert rc == _lib.ERR_BAD_ARG, (rc, msg)
    for w in words:
        assert w in msg, msg


def test_csc_checks_accept_valid_input():
    """a valid matrix passes the checks: without a GPU the call then fails for want of a device, not its input"""
    if _lib.load().icikt_device_count() > 0:
        pytest.skip("checks the no-GPU behaviour")
    for name in NAMES:
        # an empty column, a full one, explicit zeros and NaN; nnz = 0 with NULL arrays
        rc, msg = _call(name, [0, 0, 4, 6], [0, 1, 2, 3, 1, 3], [0.0, np.nan, -0.0, 1.0, 2.0, 3.0], 4, 3)
        assert rc == _lib.ERR_NO_DEVICE, (name, msg)
        rc, msg = _call(name, [0, 0, 0], None, None, 4, 2)
        assert rc == _lib.ERR_NO_DEVICE, (name, msg)


def test_malformed_sparse_object_is_refused_before_the_library():
    """colptr[C] is the number of entries the library reads: a scipy object whose arrays disagree with it
    is refused in Python, where the array lengths are known"""
    a = sp.csc_matrix((np.ones(3), np.array([0, 1, 2], dtype=np.int32), np.array([0, 1, 3])), shape=(4, 2))
    a.indptr = np.array([0, 1, 4])  # claims a fourth entry
    with pytest.raises(ValueError, match="malformed CSC"):
        _lib.run_pairs(a)


class _NoDense(sp.csc_matrix):
    """a CSC matrix that refuses to become dense"""

    def toarray(self, *a, **k):
        raise AssertionError("densified")

    def todense(self, *a, **k):
        raise AssertionError("densified")

    def __array__(self, *a, **k):
        raise AssertionError("densified")


def _sample(seed=0, n=40, C=6):
    rng = np.random.default_rng(seed)
    d = rng.normal(size=(n, C))
    d[rng.random(d.shape) < 0.6] = 0.0
    d[:, 1] = 0.0                                  # an all-implicit column
    d[:, 2] = rng.normal(size=n)                   # a fully stored column
    d[3, 3], d[4, 3], d[5, 3] = np.nan, np.inf, -2.0
    a = sp.csc_matrix(d)
    a.data[a.indices == 7] = 0.0                   # explicit zeros
    a.data[a.indices == 8] = -0.0
    return a


def _read_csc(colptr, rowidx, values, n, C):
    cp = np.array((ctypes.c_int64 * (C + 1)).from_address(colptr))
    nnz = int(cp[-1])
    ri = np.array((ctypes.c_int32 * nnz).from_address(rowidx)) if nnz else np.zeros(0, np.int32)
    va = np.array((ctypes.c_double * nnz).from_address(values)) if nnz else np.zeros(0)
    return cp, ri, va


def _dense_of(cp, ri, va, n, C):
    d = np.zeros((n, C))
    for c in range(C):
        d[ri[cp[c]:cp[c + 1]], c] = va[cp[c]:cp[c + 1]]
    return d


def _stub(monkeypatch, calls):
    """stand-ins for the matrix and completeness calls that record what they were handed"""
    real = _lib.load()

    def matrices(name):
        def f(*args):
            if name.endswith("_csc"):
                colptr, rowidx, values, n, C = args[:5]
                rest = args[5:]
                csc = _read_csc(colptr, rowidx, values, n, C)
            else:
                data, n, C, ld = args[:4]
                rest = args[4:]
                csc = None
            if "multi" in name:
                gna, ngna, opts, dev, ndev, scale_max, diag_good, n_good = rest[:8]
                mats, hist = rest[8:13], rest[13]
                pi = None
            else:
                gna, ngna, pi, pj, P, opts, scale_max, diag_good, n_good = rest[:9]
                mats, hist = rest[9:14], rest[14]
            ng = list((ctypes.c_int32 * C).from_address(n_good)) if n_good else None
            calls.append(dict(name=name, n=n, C=C, csc=csc, n_good=ng, list=bool(pi)))
            for addr in mats:
                if addr:
                    (ctypes.c_double * (C * C)).from_address(addr)[:] = [0.5] * (C * C)
            return 0
        return f

    def pairs(name):
        def f(*args):
            colptr, rowidx, values, n, C = args[:5]
            calls.append(dict(name=name, n=n, C=C, csc=_read_csc(colptr, rowidx, values, n, C)))
            if name == "icikt_pair_list_csc":
                P, outs = args[9], args[11:16]
            else:
                o = ctypes.cast(args[7], ctypes.POINTER(_lib.Opts)).contents
                P = C * (C - 1) // 2 + (C if o.include_diag else 0)
                outs = args[10:15] if "multi" in name else args[8:13]
            for addr in outs[:4]:
                (ctypes.c_double * P).from_address(addr)[:] = [0.25] * P
            (ctypes.c_int32 * P).from_address(outs[4])[:] = [0] * P
            return 0
        return f

    def completeness(*args):
        colptr, rowidx, values, n, C = args[:5]
        calls.append(dict(name="icikt_pairwise_completeness_csc", n=n, C=C, csc=_read_csc(colptr, rowidx, values, n, C)))
        mat = args[-1]
        if mat:
            (ctypes.c_double * (C * C)).from_address(mat)[:] = [1.0] * (C * C)
        return 0

    class Stub:
        icikt_matrices = staticmethod(matrices("icikt_matrices"))
        icikt_matrices_csc = staticmethod(matrices("icikt_matrices_csc"))
        icikt_matrices_multi_csc = staticmethod(matrices("icikt_matrices_multi_csc"))
        icikt_all_pairs_csc = staticmethod(pairs("icikt_all_pairs_csc"))
        icikt_all_pairs_multi_csc = staticmethod(pairs("icikt_all_pairs_multi_csc"))
        icikt_pair_list_csc = staticmethod(pairs("icikt_pair_list_csc"))
        icikt_pairwise_completeness_csc = staticmethod(completeness)

        def __getattr__(self, name):
            return getattr(real, name)

    monkeypatch.setattr(_lib, "_lib", Stub())


@pytest.mark.parametrize("global_na", [(np.nan, np.inf, 0), (np.nan, np.inf), (np.nan, -2.0)])
def test_ici_kendalltau_hands_the_csc_to_the_library(monkeypatch, global_na):
    calls = []
    _stub(monkeypatch, calls)
    a = _sample()
    dense = a.toarray()
    names = [f"s{i}" for i in range(a.shape[1])]
    ref = ik.ici_kendalltau(dense, global_na=global_na, colnames=names)
    ref_call = calls.pop()
    assert ref_call["name"] == "icikt_matrices"
    got = ik.ici_kendalltau(_NoDense(a), global_na=global_na, colnames=names)
    c = calls.pop()
    assert c["name"] == "icikt_matrices_csc" and (c["n"], c["C"]) == a.shape and not c["list"]
    cp, ri, va = c["csc"]
    assert np.array_equal(cp, a.indptr) and np.array_equal(ri, a.indices)
    assert np.array_equal(va.view(np.int64), a.data.view(np.int64))  # NaN, Inf, -0.0 as stored
    assert c["n_good"] == ref_call["n_good"]
    assert got["keep"].shape == ref["keep"].shape and np.array_equal(got["keep"], ref["keep"])
    assert got["names"] == names


def test_every_route_takes_sparse_input(monkeypatch):
    """include_only, n_gpus > 1, return_matrix=False, diag_good=False and pairwise_completeness on sparse input
    reach the *_csc entry points without a dense copy"""
    calls = []
    _stub(monkeypatch, calls)
    a = _NoDense(_sample(1))
    names = [f"s{i}" for i in range(a.shape[1])]
    ik.ici_kendalltau(a, colnames=names, include_only="s2")
    assert calls[-1]["name"] == "icikt_matrices_csc" and calls[-1]["list"]
    ik.ici_kendalltau(a, colnames=names, n_gpus=2)
    assert calls[-1]["name"] == "icikt_matrices_multi_csc"
    r = ik.ici_kendalltau(a, colnames=names, return_matrix=False, diag_good=False)
    assert calls[-1]["name"] == "icikt_all_pairs_csc" and len(r["cor"]["raw"]) == 21
    r = ik.ici_kendalltau(a, colnames=names, return_matrix=False, diag_good=True)
    assert calls[-1]["name"] == "icikt_all_pairs_csc" and len(r["cor"]["raw"]) == 21  # 15 pairs + the diagonal
    r = ik.ici_kendalltau(a, colnames=names, check_timing=True)
    assert calls[-1]["name"] == "icikt_pair_list_csc" and r["value"][1] == 15
    r = _lib.run_pairs(a, (), devices=[0, 1])
    assert calls[-1]["name"] == "icikt_all_pairs_multi_csc" and r["raw"].shape == (15,)
    _lib.run_pairs(a, (), pi=[0], pj=[1])
    assert calls[-1]["name"] == "icikt_pair_list_csc"
    m = ik.pairwise_completeness(a, colnames=names)
    assert calls[-1]["name"] == "icikt_pairwise_completeness_csc" and m.shape == (6, 6)
    for c in calls:
        cp, ri, va = c["csc"]
        assert np.array_equal(_dense_of(cp, ri, va, *a.shape), sp.csc_matrix(a).toarray(), equal_nan=True)


def test_non_canonical_input_arrives_canonical(monkeypatch):
    """unsorted rows and duplicate entries (summed, as toarray() sums them) reach the library in canonical
    form; the caller's object is not modified.  COO and CSR input are converted."""
    calls = []
    _stub(monkeypatch, calls)
    indptr = np.array([0, 3, 3, 7])
    indices = np.array([2, 0, 2, 5, 1, 5, 0], dtype=np.int32)
    data = np.array([1.0, 2.0, 3.0, 4.0, 5.0, -6.0, 7.0])
    a = sp.csc_matrix((data.copy(), indices.copy(), indptr.copy()), shape=(6, 3))
    assert not a.has_canonical_format
    want = a.toarray()
    for x in (a, sp.coo_matrix(want), sp.csr_matrix(want), sp.csc_array(a)):
        _lib.run_pairs(x, ())
        cp, ri, va = calls[-1]["csc"]
        assert np.array_equal(_dense_of(cp, ri, va, 6, 3), want)
        for c in range(3):
            rows = ri[cp[c]:cp[c + 1]]
            assert np.all(np.diff(rows) > 0), rows
    assert np.array_equal(a.indices, indices) and np.array_equal(a.data, data) and np.array_equal(a.indptr, indptr)
    _lib.pairwise_completeness(a, (np.nan, 0.0))
    cp, ri, va = calls[-1]["csc"]
    assert np.array_equal(cp, [0, 2, 2, 5]) and np.array_equal(ri, [0, 2, 0, 1, 5])
    assert np.array_equal(va, [2.0, 4.0, 7.0, 5.0, -2.0])


def test_sparse_argument_checks():
    a = _sample()
    with pytest.raises(ValueError, match="Colnames of `data_matrix` must be be specified."):
        ik.ici_kendalltau(a)
    with pytest.raises(ValueError, match="has 5 entries"):
        ik.ici_kendalltau(a, colnames=list("abcde"))
    with pytest.raises(TypeError, match="must be a numeric type"):
        ik.ici_kendalltau(a.astype(bool), colnames=list("abcdef"))


@pytest.mark.parametrize("where", ["early", "late", "both"])
def test_csc_checks_of_a_large_matrix_name_the_first_bad_column(where):
    """above a million entries the row scan is split over host threads; the message still names the first bad
    column, whichever thread finds it"""
    n, C, per = 4096, 1024, 2048  # 2 M entries
    rng = np.random.default_rng(3)
    rows = np.concatenate([np.sort(rng.choice(n, per, replace=False)) for _ in range(C)]).astype(np.int32)
    colptr = np.arange(C + 1, dtype=np.int64) * per
    values = np.ones(rows.size)
    if where in ("early", "both"):
        rows[5 * per + 7] = rows[5 * per + 6]       # column 5 repeats a row
    if where in ("late", "both"):
        rows[900 * per + 3] = n                     # column 900: row out of range
    rc, msg = _call("icikt_all_pairs_csc", colptr, rows, values, n, C)
    assert rc == _lib.ERR_BAD_ARG, msg
    if where == "late":
        assert f"row {n} of column 900" in msg, msg
    else:
        assert "column 5 repeat row" in msg, msg
