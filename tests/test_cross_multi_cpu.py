"""The cross calls over several devices (icikt_cross_pairs_multi, icikt_cross_edges_multi, icikt_cross_topk_multi)
without a GPU: every argument check that runs before any device is touched, with the single-device cross calls'
messages, and the Python routing with a stand-in for the library."""
import ctypes

import numpy as np
import pytest
import scipy.sparse as sp

import icikendalltau_b200 as ik
from icikendalltau_b200 import _lib
from tests import test_cross_cpu as X

NAMES = ("icikt_cross_pairs_multi", "icikt_cross_edges_multi", "icikt_cross_topk_multi")


class MultiArgs(X.Args):
    """valid arguments of one multi-device entry point; tests change one thing"""

    def __init__(self, **kw):
        super().__init__(**kw)
        self.devices = np.array([0, 0, 1], dtype=np.int32)
        self.n_devices = 3
        self.use_devices = True

    def call(self, name):
        L = _lib.load()
        x = ctypes.byref(self.xi) if self.x_ref else None
        y = ctypes.byref(self.yi) if self.y_ref else None
        lead = (x, y, self.n, None, 0, ctypes.byref(self.opts),
                self.devices.ctypes.data if self.use_devices else None, self.n_devices)
        mx = ctypes.c_double(7.0)
        if name == "icikt_cross_pairs_multi":
            rc = L.icikt_cross_pairs_multi(*lead, self.raw.ctypes.data if self.raw is not None else None, None, None,
                                           None, None, ctypes.byref(mx), None)
        elif name == "icikt_cross_edges_multi":
            rc = L.icikt_cross_edges_multi(*lead, ctypes.byref(self.filter) if self.use_filter else None,
                                           ctypes.byref(self.out) if self.use_out else None, ctypes.byref(mx), None)
        else:
            rc = L.icikt_cross_topk_multi(*lead, self.k, self.by, 1,
                                          ctypes.byref(self.x_side) if self.sides[0] else None,
                                          ctypes.byref(self.y_side) if self.sides[1] else None, ctypes.byref(mx), None)
        self.mx = mx.value
        return rc, L.icikt_last_error().decode()


DEVICES = {
    "n_devices_zero": (lambda a: setattr(a, "n_devices", 0), "n_devices must be 1..16"),
    "n_devices_negative": (lambda a: setattr(a, "n_devices", -1), "n_devices must be 1..16"),
    "n_devices_17": (lambda a: (setattr(a, "devices", np.zeros(17, dtype=np.int32)), setattr(a, "n_devices", 17)),
                     "n_devices must be 1..16"),
}
ALL = {**X.ALL, **DEVICES}
CASES = ([("icikt_cross_pairs_multi", c) for c in sorted({**X.COMMON, **X.PAIRS_ONLY, **DEVICES})] +
         [("icikt_cross_edges_multi", c) for c in sorted({**X.COMMON, **X.WHOLE, **X.EDGES_ONLY, **DEVICES})] +
         [("icikt_cross_topk_multi", c) for c in sorted({**X.COMMON, **X.WHOLE, **X.TOPK_ONLY, **DEVICES})])


def test_entry_points_exported():
    assert set(NAMES) <= set(_lib.EXPORTS)
    L = _lib.load()
    for name in NAMES:
        single = getattr(L, name[:-len("_multi")]).argtypes
        assert getattr(L, name).argtypes == single[:6] + [_lib._ip, ctypes.c_int32] + single[6:]


@pytest.mark.parametrize("name,case", CASES)
def test_refused_arguments_before_any_device_work(name, case):
    a = MultiArgs()
    change, words = ALL[case]
    change(a)
    rc, msg = a.call(name)
    assert rc == _lib.ERR_BAD_ARG, (rc, msg)
    assert words in msg, msg
    assert a.untouched() and a.mx == 7.0
    if name == "icikt_cross_edges_multi" and a.use_out:
        assert a.out.value is None  # *out cleared


@pytest.mark.parametrize("name", NAMES)
def test_refusal_messages_match_the_single_device_call(name):
    for case in sorted(X.COMMON):
        one, many = X.Args(), MultiArgs()
        X.ALL[case][0](one)
        X.ALL[case][0](many)
        assert one.call(name[:-len("_multi")]) == many.call(name), case


@pytest.mark.skipif(X._has_gpu(), reason="checks the no-GPU behaviour")
@pytest.mark.parametrize("name", NAMES)
def test_no_device(name):
    for devices, n_devices in ((np.array([0, 0, 1], dtype=np.int32), 3), (None, 2), (np.array([0], dtype=np.int32), 1),
                               (np.zeros(16, dtype=np.int32), 16)):
        a = MultiArgs()
        a.devices, a.n_devices, a.use_devices = devices, n_devices, devices is not None
        rc, msg = a.call(name)
        assert rc == _lib.ERR_NO_DEVICE, (n_devices, msg)
        assert a.untouched()
    a = MultiArgs()  # CSC on both sides, a slice of the pairs, one side of the lists
    a.xcsc = (np.array([0, 1, 3, 4], dtype=np.int64), np.array([1, 2, 5, 4], dtype=np.int32), np.ones(4))
    a.xi = _lib.Input(3, None, 0, *(v.ctypes.data for v in a.xcsc))
    a.ycsc = (np.array([0, 1, 2, 3, 4], dtype=np.int64), np.array([1, 2, 3, 4], dtype=np.int32), np.ones(4))
    X._bad_csc(a)
    a.sides = (False, True)
    if name == "icikt_cross_pairs_multi":
        a.opts.pair_lo, a.opts.pair_hi = 3, 12
    rc, msg = a.call(name)
    assert rc == _lib.ERR_NO_DEVICE, msg
    if name == "icikt_cross_pairs_multi":  # an empty slice still needs the device, as on one device
        a.opts.pair_lo, a.opts.pair_hi = 5, 5
        assert a.call(name)[0] == _lib.ERR_NO_DEVICE


# ---------------------------------------------------------------- Python routing
def _stub(monkeypatch, calls):
    """stand-ins for the cross calls that record their name and the devices they were handed"""
    real = _lib.load()

    def call(name):
        def f(*args):
            rec = dict(name=name, Cx=args[0]._obj.C, Cy=args[1]._obj.C)
            if name.endswith("_multi"):
                dev, ndev = args[6], args[7]
                rec["devices"] = list((ctypes.c_int32 * ndev).from_address(dev)) if ndev else []
            calls.append(rec)
            return 0
        return f

    class Stub:
        def __getattr__(self, name):
            if name.startswith("icikt_cross_"):
                return call(name)
            if name == "icikt_edges_count":
                return lambda h: 0
            if name == "icikt_edges_copy":
                return lambda *a: 0
            if name == "icikt_edges_free":
                return lambda h: None
            return getattr(real, name)

    monkeypatch.setattr(_lib, "_lib", Stub())


def test_run_cross_routes(monkeypatch):
    calls = []
    _stub(monkeypatch, calls)
    rng = np.random.default_rng(3)
    x, y = rng.normal(size=(30, 2)), rng.normal(size=(30, 5))
    ys = sp.random(30, 5, density=0.4, format="csc", random_state=4)
    for run, base in ((lambda a, b, **kw: ik.run_cross(a, b, (), **kw), "icikt_cross_pairs"),
                      (lambda a, b, **kw: ik.run_cross_edges(a, b, (), 0.5, **kw), "icikt_cross_edges"),
                      (lambda a, b, **kw: ik.run_cross_topk(a, b, (), 3, side="x", **kw), "icikt_cross_topk")):
        run(x, y, devices=[0, 1, 0])
        assert calls[-1] == dict(name=base + "_multi", Cx=2, Cy=5, devices=[0, 1, 0])
        run(x, ys, devices=(2,))
        assert calls[-1] == dict(name=base + "_multi", Cx=2, Cy=5, devices=[2])
        run(ys, x, devices=range(4))
        assert calls[-1] == dict(name=base + "_multi", Cx=5, Cy=2, devices=[0, 1, 2, 3])
        run(x, y)
        assert calls[-1] == dict(name=base, Cx=2, Cy=5)


def test_api_cross_calls_still_refuse_several_gpus(monkeypatch):
    calls = []
    _stub(monkeypatch, calls)
    rng = np.random.default_rng(5)
    x, y = rng.normal(size=(30, 2)), rng.normal(size=(30, 4))
    xn, yn = ["a", "b"], list("cdef")
    with pytest.raises(ValueError, match="n_gpus must be 1"):
        ik.ici_kendalltau_cross(x, y, xnames=xn, ynames=yn, n_gpus=2)
    with pytest.raises(ValueError, match="n_gpus must be 1"):
        ik.ici_kendalltau_cross_topk(x, y, 2, xnames=xn, ynames=yn, n_gpus=2)
    assert calls == []
