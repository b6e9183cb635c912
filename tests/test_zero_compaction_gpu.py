"""The pair kernel's handling of the other column's lowest-rank (zero) keys -- the rows missing in y, which
pass A sees as zero keys (DESIGN.md section 2, round 4): counts bit for bit against the CPU oracle and the
one-thread-per-pair kernel on left-censored data like the benchmark's target, columns without missing values,
the absorbed case (missing rows tie with the minimum), small x tie groups holding y-missing rows, nearly
all-missing columns, and numbers of y-present rows just below, on and just above multiples of a thread's
range and of 8; through the all-pairs, pair-list and edges calls."""
import os

import numpy as np
import pytest

import icikendalltau_b200 as ik
from icikendalltau_b200 import _lib, synth
from oracle import oracle as O


def oracle_counts(x, pi, pj):
    return O.pair_loop(np.array(x, copy=True), pi, pj, ncore=os.cpu_count() or 1, want_counts=True)


def check(x, with_oracle=True):
    C = x.shape[1]
    got = ik.run_pairs(x, (), want_counts=True)
    naive = ik.run_pairs(x, (), want_counts=True, kernel=_lib.KERNEL_NAIVE)
    assert np.array_equal(got["status"], naive["status"])
    assert np.array_equal(got["counts"], naive["counts"])
    if with_oracle:
        pi, pj = O.setup_comparisons(C, None, True)
        ref = oracle_counts(x, pi, pj)
        assert np.array_equal(got["status"], ref["status"])
        ok = ref["status"] == 0
        assert np.array_equal(got["counts"][ok], ref["counts"][ok])
    return got


def censored(n, C, missing, seed, ties=0):
    """C columns of n rows; column c has missing[c] missing rows (NaN), the rest distinct values
    (or values rounded to `ties` levels)."""
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((n, C))
    if ties:
        x = np.round(x * ties)
    for c in range(C):
        x[rng.permutation(n)[:missing[c]], c] = np.nan
    return np.asfortranarray(x)


@pytest.mark.gpu
def test_target_like():
    x, _ = synth.make("target", n=20000, C=6)
    check(x)


@pytest.mark.gpu
def test_no_missing_values():
    check(censored(5000, 5, [0] * 5, seed=1))


@pytest.mark.gpu
def test_absorbed_minimum():
    """values so large that min - 0.1 == min: the missing rows share the column's lowest rank"""
    rng = np.random.default_rng(2)
    x = 1e17 + 1024.0 * rng.integers(0, 3000, size=(4000, 5)).astype(np.float64)
    x[rng.random(x.shape) < 0.25] = np.nan
    x[:, 1] = rng.standard_normal(4000)  # a column that is not absorbed
    check(np.asfortranarray(x))


@pytest.mark.gpu
def test_small_x_ties_with_y_missing_rows():
    check(censored(6000, 5, [1500, 900, 2500, 0, 3000], seed=3, ties=40))
    check(censored(6000, 5, [1500, 900, 2500, 10, 3000], seed=4, ties=400))


@pytest.mark.gpu
def test_nearly_all_missing():
    n = 8000
    check(censored(n, 5, [n - 2, n - 3, n - 40, n - 700, 100], seed=5))


@pytest.mark.gpu
@pytest.mark.parametrize("n", [3000, 20000])
def test_lengths_around_range_multiples(n, monkeypatch):
    """y's present rows (pass A's length without the zero keys) just below, on and just above multiples of
    the thread range R of the launch shape and of 8.  The shape is the one of a large job, pinned with
    ICIKT_WARPS: these few pairs would otherwise plan a wider one with another R."""
    shape = _lib.launch_shape(n, 0)
    monkeypatch.setenv("ICIKT_WARPS", str(shape["warps"]))
    _lib.release_workspace()
    assert _lib.launch_shape(n, 0) == shape
    R = 8 * shape["runs"]
    lens = set()
    for m in (R, 8, 32 * R):
        for k in (1, 2, 7, n // m - 1):
            for d in (-1, 0, 1):
                v = k * m + d
                if 2 <= v <= n - 1:
                    lens.add(v)
    lens = sorted(lens)
    for i in range(0, len(lens), 4):
        part = lens[i:i + 4]
        miss = [n - v for v in part] + [n // 4]
        check(censored(n, len(miss), miss, seed=100 + i), with_oracle=(n <= 3000))
    _lib.release_workspace()


@pytest.mark.gpu
def test_pair_list_and_edges():
    x, _ = synth.make("target", n=20000, C=8)
    full = ik.run_pairs(x, (), want_counts=True)
    pi, pj = O.setup_comparisons(8, None, True)
    sel = np.arange(0, len(pi), 3)
    lst = ik.run_pairs(x, (), pi=np.asarray(pi)[sel], pj=np.asarray(pj)[sel], want_counts=True)
    assert np.array_equal(lst["counts"], full["counts"][sel])
    assert np.array_equal(lst["raw"], full["raw"][sel])
    e = ik.run_edges(x, (), min_abs_cor=0.0)
    m = ~np.isnan(full["raw"])
    assert np.array_equal(np.sort(e["raw"]), np.sort(full["raw"][m]))
