"""The sign-vector reference (tests/sign_reference.py) against the CPU oracle, before any GPU test relies on it, and
icikt_pair_from_index against an exact integer inverse of the combn order up to INT32_MAX columns."""
import math
import os

import numpy as np
import pytest

from icikendalltau_b200 import _lib
from oracle import oracle as O
from tests import sign_reference as SR


def _oracle(x, pi, pj, persp):
    return O.pair_loop(x, pi, pj, perspective=persp, ncore=os.cpu_count() or 1, want_counts=True)


def _data(n, C, kind, seed):
    rng = np.random.default_rng(seed)
    x = rng.normal(size=(n, 1)) + rng.normal(size=(n, C)) * 0.8
    if kind in ("ties", "ties_censored", "ties_random_na"):
        x = np.round(x * 1.5)
    if kind in ("censored", "ties_censored"):  # left-censored: the lowest values of the matrix are missing
        x = np.where(x <= np.quantile(x, 0.3), np.nan, x)
    if kind in ("random_na", "ties_random_na"):
        x[rng.random(x.shape) < 0.25] = np.nan
    if kind == "degenerate" and C >= 6:
        x[:, 0] = np.nan                   # all missing
        x[:, 1] = 2.0                      # constant
        x[:, 2] = np.where(rng.random(n) < 0.5, np.nan, 3.0)  # one value and missing rows
        x[: max(n - 1, 0), 3] = np.nan     # a single present row
        x[:, 4] = np.where(np.arange(n) < n // 2, np.nan, x[:, 4])
        x[:, 5] = np.where(np.arange(n) < n // 2, np.nan, x[:, 5])  # the same missing rows as column 4
    return np.asfortranarray(x)


KINDS = ("plain", "ties", "censored", "random_na", "ties_censored", "ties_random_na", "degenerate")


@pytest.mark.parametrize("persp", ["global", "local"])
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("n", [2, 3, 5, 17, 40, 64])
def test_sign_reference_matches_oracle(n, kind, persp):
    C = 9
    x = _data(n, C, kind, seed=1000 * n + KINDS.index(kind))
    pi, pj = O.setup_comparisons(C, None, False)  # every pair and the diagonal
    ref = _oracle(x, pi, pj, persp)
    st = SR.pairs(SR.Features(x), pi, pj, persp)
    counts, status = SR.counts_matrix(st)
    assert np.array_equal(status, ref["status"]), f"status {status} vs {ref['status']}"
    ok = status == 0
    for k, name in enumerate(SR.COUNT_NAMES):
        assert np.array_equal(counts[ok, k], ref["counts"][ok, k]), name
    # the whole matrix of products gives the same pairs as the listed ones
    F = SR.Features(x)
    blk = SR.block(F, F, persp)
    for name in SR.COUNT_NAMES + ("status",):
        assert np.array_equal(blk[name][pi, pj], st[name]), name
    for name in ("raw", "taumax"):
        a, b = st[name][ok], ref[name][ok]
        np.testing.assert_allclose(a, b, rtol=1e-12, atol=0, err_msg=name)
        assert np.array_equal(blk[name][pi, pj], st[name], equal_nan=True), name


def test_sign_reference_tie_free_raw_is_s_over_tot():
    """on complete tie-free columns taumax is 1 and raw = S / K exactly, what the walks over D1 rely on"""
    rng = np.random.default_rng(5)
    n = 40
    x = np.argsort(rng.random((n, 30)), axis=0).astype(np.float64)
    F = SR.Features(x)
    b = SR.block(F, F)
    K = n * (n - 1) // 2
    off = ~np.eye(30, dtype=bool)
    assert (b["taumax"][off] == 1.0).all()
    assert np.array_equal(b["raw"][off], b["S"][off] / K)


# ---------------------------------------------------------------- icikt_pair_from_index at large C
INT32_MAX = 2 ** 31 - 1


def _guess(C, index):
    """the float guess of icikt_pair_from_index before its fix-up loops, in the same IEEE double operations"""
    b = 2.0 * C - 1.0
    d = b * b - 8.0 * float(index)
    if not d >= 0.0:
        return None
    return max(0, min(int((b - math.sqrt(d)) / 2.0), C - 2))


def _indices(C, rng):
    """every row start +- 1 of the first and last 64 rows, row starts and row ends of random rows, random indices"""
    ptri = C * (C - 1) // 2
    rows = list(range(min(64, C - 1))) + list(range(max(0, C - 65), C - 1))
    rows += [int(r) for r in rng.integers(0, C - 1, 64)]
    out = set()
    for r in rows:
        s = SR.row_start(C, r)
        out.update((s - 1, s, s + 1, s + C - 2 - r))
    out.update(int(v) for v in rng.integers(0, ptri, 256))
    out.update((0, ptri - 1, 2 ** 31 - 1, 2 ** 31, 2 ** 32 - 1, 2 ** 32, 2 ** 32 + 1))
    return sorted(v for v in out if 0 <= v < ptri)


@pytest.mark.parametrize("C", [2, 3, 65600, 92700, 2 ** 16 + 1, 3 * 2 ** 20 + 7, 2 ** 30 + 3, INT32_MAX - 1,
                               INT32_MAX])
def test_pair_from_index_exact_to_int32_max(C):
    rng = np.random.default_rng(C)
    worst = 0
    for p in _indices(C, rng):
        want = SR.pair_index(C, p)
        assert _lib.pair_from_index(C, p) == want, f"C={C} p={p}"
        assert want[0] < want[1] < C and SR.row_start(C, want[0]) + want[1] - want[0] - 1 == p
        g = _guess(C, p)
        assert g is not None, f"C={C} p={p}: negative discriminant"
        worst = max(worst, abs(g - want[0]))
    # the fix-up loops step from the float guess to the row: a few steps, not a walk over the rows
    assert worst <= 32, f"C={C}: the float guess is {worst} rows off"
    ptri = C * (C - 1) // 2
    for d in range(min(C, 3)):
        assert _lib.pair_from_index(C, ptri + d, include_diag=True) == (d, d)
    for bad in (ptri, -1):
        with pytest.raises(_lib.IciktError):
            _lib.pair_from_index(C, bad)


def test_pair_index_inverse_is_combn_order():
    for C in (2, 3, 7, 50):
        iu = np.triu_indices(C, 1)
        for p in range(C * (C - 1) // 2):
            assert SR.pair_index(C, p) == (iu[0][p], iu[1][p])
        assert SR.pair_index(C, C * (C - 1) // 2 + C - 1) == (C - 1, C - 1)


def test_run_pairs_refuses_a_slice_over_several_devices():
    """the multi-device per-pair call covers the whole pair order: a slice must be refused before any buffer is
    sized for it (the library would write every pair)"""
    x = np.zeros((4, 5))
    with pytest.raises(ValueError, match="pair_lo"):
        _lib.run_pairs(x, (), devices=[0, 0], pair_lo=1, pair_hi=3)
