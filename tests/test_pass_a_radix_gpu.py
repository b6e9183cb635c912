"""Pass A's radix-16 levels against the oracle's counts, bit for bit: bit counts L one below, at and one above
each 4-bit boundary of the level structure, lengths on both sides of the length range that takes radix levels,
launch tiers 0, 1 and 2, the complete-observations mode, and pairs with and without y's lowest-rank rows left
out of pass A."""
import numpy as np
import pytest

import icikendalltau_b200 as ik
from icikendalltau_b200 import _lib
from tests.test_gpu_parity import _oracle_complete
from tests.test_launch_variants_gpu import (censored, check, checked_stats, distinct_col, grouped_col, ordered_pairs,
                                            tier2_matrix, tier_of, with_missing)
from tests.test_pass_a_levels_gpu import check as check_levels, columns

RADIX_LO, RADIX_HI = 8193, 27648  # the lengths that take radix levels (checked by tests/test_pass_a_radix_cpu.py)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [RADIX_LO - 1, RADIX_LO, 20000, RADIX_HI, RADIX_HI + 1])
@pytest.mark.parametrize("L", [7, 8, 9, 11, 12, 13, 14, 15])
def test_counts_at_structure_changes(n, L):
    K = (1 << (L - 1)) + 1  # exactly L bits
    if K > n:
        pytest.skip("more ranks than rows")
    assert _lib.pass_a_radix(n) == (RADIX_LO <= n <= RADIX_HI)
    lead = (0, 257, 1025)[(n + L) % 3]
    check_levels(columns(n, K, lead if K + lead <= n else 0, 3, seed=n + L))


def tier1_matrix(n, seed):
    """8 large tie groups of 1 000 rows in one column (8 x K <= 16 n for every K: the large-group sort, no pass B)
    beside tie-free, left-censored and heavily tied columns"""
    rng = np.random.default_rng(seed)
    names = ["G", "GL", "D", "N", "R"]
    cols = [grouped_col(rng, n, 8, 1000), grouped_col(rng, n, 8, 1000, n_na=n // 5), distinct_col(rng, n, n // 2),
            with_missing(rng, rng.standard_normal(n), n // 4), np.round(rng.standard_normal(n))]
    return names, np.asfortranarray(np.column_stack(cols))


def check_complete(names, x):
    keep = [k for k, nm in enumerate(names) if nm not in ("HA", "DA")]  # absorbed columns: host path (status 9)
    xc = np.asfortranarray(x[:, keep])
    pi, pj = ordered_pairs(len(keep))
    got = ik.run_pairs(xc, (), pi=pi, pj=pj, perspective="complete", want_counts=True)
    ref = _oracle_complete(xc, pi, pj)
    np.testing.assert_array_equal(got["status"], ref["status"])
    ok = ref["status"] == 0
    np.testing.assert_array_equal(got["counts"][ok, :6], ref["counts"][ok, :6])
    np.testing.assert_allclose(got["raw"][ok], ref["raw"][ok], rtol=1e-12, atol=0)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [20000, RADIX_HI])
@pytest.mark.parametrize("tier", [1, 2])
def test_tiers_and_complete_observations(n, tier):
    names, x = tier1_matrix(n, seed=n) if tier == 1 else tier2_matrix(n, 40, 200, seed=n)
    assert tier_of(checked_stats(x), n) == tier and _lib.pass_a_radix(n)
    pi, pj = ordered_pairs(len(names))
    check(x, pi, pj, what=f"n={n} tier {tier}")
    check_complete(names, x)


@pytest.mark.gpu
def test_compacted_and_uncompacted_pairs():
    """left-censored columns whose missing counts run from none to a whole warp's ranges and more"""
    n = 20000
    missing = [0, 1, 255, 4000, 5000, 5119, 5120, 5121, 9000]
    x = censored(n, missing, seed=5)
    st = checked_stats(x)
    assert tier_of(st, n) == 0 and _lib.pass_a_radix(n)
    pi, pj = ordered_pairs(len(missing))
    check(x, pi, pj, what="censored")
