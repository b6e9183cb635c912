"""The refusals of the ten per-pair and matrix entry points (icikt_all_pairs, icikt_all_pairs_multi, icikt_pair_list,
icikt_matrices, icikt_matrices_multi and their CSC twins), one bad argument at a time: the return code and the text of
icikt_last_error().  Without a GPU, a call whose arguments pass every host-side check fails with ICIKT_ERR_NO_DEVICE
(there is no CPU fallback); those cases are skipped where a device exists."""
import ctypes

import numpy as np
import pytest
import scipy.sparse as sp

from icikendalltau_b200 import _lib


def _has_gpu():
    try:
        return _lib.load().icikt_device_count() > 0
    except Exception:
        return False


NO_DEVICE = (_lib.ERR_NO_DEVICE, "no CUDA device available (this library has no CPU fallback)")
BAD = _lib.ERR_BAD_ARG
N, C = 20, 5


def _call(name, n=N, C=C, ld=None, data=True, raw=True, pi=(0, 1), pj=(2, 3), P=None, devices=(0,), n_devices=None,
          opts=None, csc_bad=False):
    """one call of entry point `name` with the given arguments; (rc, message)"""
    L = _lib.load()
    cols = max(C, 1) if C < 1 << 20 else 1
    if name.endswith("_csc"):
        m = _lib.CSC(sp.random(n, cols, density=0.5, format="csc", random_state=1))
        if csc_bad:
            m.rowidx[0] = n  # a row outside [0, n) in column 0
        lead = (m.colptr.ctypes.data, m.rowidx.ctypes.data, m.values.ctypes.data, n, C)
    else:
        x = np.asfortranarray(np.random.default_rng(0).normal(size=(n, cols)))
        lead = (x.ctypes.data if data else None, n, C, n if ld is None else ld)
    o = opts if opts is not None else _lib.make_opts()
    out = np.zeros(8 * (N * N + N), dtype=np.float64)
    mx, t = ctypes.c_double(), _lib.Timings()
    a_raw = out.ctypes.data if raw else None
    ia = None if pi is None else np.ascontiguousarray(pi, dtype=np.int32)
    ja = None if pj is None else np.ascontiguousarray(pj, dtype=np.int32)
    p_args = (None if ia is None else ia.ctypes.data, None if ja is None else ja.ctypes.data,
              (0 if ia is None else ia.size) if P is None else P)
    dev = np.ascontiguousarray(devices, dtype=np.int32)
    d_args = (dev.ctypes.data, len(devices) if n_devices is None else n_devices)
    fn = getattr(L, name)
    base = name.replace("_csc", "")
    if base in ("icikt_all_pairs", "icikt_all_pairs_multi", "icikt_pair_list"):
        mid = {"icikt_all_pairs": (), "icikt_all_pairs_multi": d_args, "icikt_pair_list": ()}[base]
        pre = p_args if base == "icikt_pair_list" else ()
        rc = fn(*lead, None, 0, *pre, ctypes.byref(o), *mid, a_raw, None, None, None, None, None, ctypes.byref(mx),
                ctypes.byref(t))
    elif base == "icikt_matrices":
        mats = (a_raw, None, None, None, None)
        rc = fn(*lead, None, 0, *p_args, ctypes.byref(o), 1, 1, None, *mats, None, ctypes.byref(mx), ctypes.byref(t))
    else:
        mats = (a_raw, None, None, None, None)
        rc = fn(*lead, None, 0, ctypes.byref(o), *d_args, 1, 1, None, *mats, None, ctypes.byref(mx), ctypes.byref(t))
    return rc, L.icikt_last_error().decode()


ALL = C * (C - 1) // 2  # the pairs of C columns without the diagonal
_opts = _lib.make_opts


def _cases():
    """(entry point, arguments, expected (rc, message))"""
    too_long = (_lib.ERR_TOO_LONG, "n exceeds icikt_max_n()")
    n_c = (BAD, "n and C must be >= 1")
    upload = (BAD, "bad upload arguments")
    rng = (BAD, "pair_lo/pair_hi out of range")
    families = {
        "icikt_all_pairs": dict(pi=None, pj=None),
        "icikt_all_pairs_multi": dict(pi=None, pj=None, devices=(0, 0)),
        "icikt_pair_list": dict(),
        "icikt_matrices": dict(pi=None, pj=None),
        "icikt_matrices_multi": dict(pi=None, pj=None, devices=(0, 0)),
    }
    for fam, base in families.items():
        matrix = fam.startswith("icikt_matrices")
        multi = fam.endswith("_multi")
        for name in (fam, fam + "_csc"):
            csc = name.endswith("_csc")

            def case(label, expect, **kw):
                return pytest.param(name, dict(base, **kw), expect, id=f"{name}-{label}")

            yield case("valid", NO_DEVICE)
            yield case("n_zero", n_c, n=0)
            yield case("C_zero", n_c, C=0)
            yield case("n_too_long", too_long, n=_lib.load().icikt_max_n() + 1)
            if csc:
                yield case("csc_row_out_of_range", (BAD, f"CSC input: row {N} of column 0 is outside [0, {N})"),
                           csc_bad=True)
            else:
                yield case("ld_below_n", upload, ld=N - 1)
                yield case("too_many_columns", (BAD, "too many columns"), C=1 << 31)
                data_msg = "data must not be NULL" if matrix and multi else "data and raw must not be NULL"
                yield case("data_null", (BAD, data_msg), data=False)
            yield case("raw_null", NO_DEVICE if matrix else (BAD, "data and raw must not be NULL"), raw=False)
            if multi:
                lim = 16 if matrix else 64
                msg = (BAD, f"n_devices must be 1..{lim}")
                yield case("n_devices_zero", msg, n_devices=0)
                yield case("n_devices_over", msg, devices=(0,) * (lim + 1))
                yield case("one_device", NO_DEVICE, devices=(0,))
                if not csc:
                    yield case("one_device_ld_below_n", upload, devices=(0,), ld=N - 1)
                yield case("pair_range_ignored", NO_DEVICE, opts=_opts(pair_lo=ALL + 3, pair_hi=ALL + 1))
            elif fam == "icikt_all_pairs":
                yield case("pair_range", NO_DEVICE, opts=_opts(pair_lo=1, pair_hi=4))
                yield case("pair_hi_beyond", rng, opts=_opts(pair_lo=0, pair_hi=ALL + 1))
                yield case("pair_lo_above_hi", rng, opts=_opts(pair_lo=4, pair_hi=2))
                yield case("pair_lo_negative", rng, opts=_opts(pair_lo=-1, pair_hi=2))
                yield case("pair_hi_without_lo", rng, opts=_opts(pair_lo=3, pair_hi=0))
            elif fam == "icikt_pair_list":
                yield case("pi_null", (BAD, "pi and pj must not be NULL"), pi=None)
                yield case("pj_null", (BAD, "pi and pj must not be NULL"), pj=None)
                yield case("empty_list", (BAD, "empty pair list"), P=0)
                yield case("pair_index_out_of_range", NO_DEVICE, pi=(0, C))
            else:  # icikt_matrices
                yield case("pj_null", (BAD, "pi and pj must both be given"), pi=(0, 1), pj=None)
                yield case("pi_null", (BAD, "pi and pj must both be given"), pi=None, pj=(0, 1))
                yield case("pair_list", NO_DEVICE, pi=(0, 1), pj=(2, 3))
                yield case("empty_list", (BAD, "empty pair list"), pi=(0, 1), pj=(2, 3), P=0)
                yield case("pair_range", (BAD, "matrix output needs the whole pair order on one device"),
                           opts=_opts(pair_lo=1, pair_hi=4))


@pytest.mark.parametrize("name,kw,expect", list(_cases()))
def test_refusal(name, kw, expect):
    if expect[0] == _lib.ERR_NO_DEVICE and _has_gpu():
        pytest.skip("checks the no-GPU behaviour")
    rc, msg = _call(name, **kw)
    assert (rc, msg) == expect
