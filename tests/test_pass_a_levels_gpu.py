"""Pass A's levels against the oracle's counts, bit for bit: rank counts K that give an odd and an even
number of bits L, and fewer than the four bits of the count-only low-nibble level; leading blocks of rows
missing in both columns that end inside, on and just past a thread's range; lengths on both sides of
the fused column kernel's limit, the global-scratch limit and the in-place threshold, so that every
producer of the per-column constant and both forms of pass A run."""
import os

import numpy as np
import pytest

import icikendalltau_b200 as ik
from oracle import oracle as O

def columns(n, K, lead, C, seed):
    """C columns of n rows with exactly min(K, n - lead) distinct values (heavy ties for small K); the
    first `lead` rows are missing in every column, so they open every pair's sequence as one block."""
    rng = np.random.default_rng(seed)
    x = rng.integers(0, K, size=(n, C)).astype(np.float64)
    k = min(K, n - lead)
    for c in range(C):
        x[lead:lead + k, c] = rng.permutation(k)
    x[lead:] = x[lead:][rng.permutation(n - lead)]
    x[:lead] = np.nan
    return np.asfortranarray(x)


def check(x):
    got = ik.run_pairs(x, (), want_counts=True)
    pi, pj = O.setup_comparisons(x.shape[1], None, True)
    ref = O.pair_loop(np.array(x, copy=True), pi, pj, ncore=os.cpu_count() or 1, want_counts=True)
    assert np.array_equal(got["status"], ref["status"])
    ok = ref["status"] == 0
    assert ok.any()
    assert np.array_equal(got["counts"][ok], ref["counts"][ok])
    m = ~np.isnan(ref["raw"])
    assert np.array_equal(got["raw"][m], ref["raw"][m])


LENGTHS = [8191, 8193, 22527, 22529, 54273, 65535]
RANKS = [2, 3, 5, 16, 17, 1 << 14, (1 << 14) + 1, 65535]


@pytest.mark.gpu
@pytest.mark.parametrize("n", LENGTHS)
@pytest.mark.parametrize("K", RANKS)
def test_counts_over_bit_widths(n, K):
    if K > n:
        pytest.skip("more ranks than rows")
    lead = (0, 257, 4096)[(n + K) % 3]
    check(columns(n, K, lead if K + lead <= n else 0, 3, seed=n * 7 + K))


@pytest.mark.gpu
@pytest.mark.parametrize("lead", [255, 256, 257, 767, 768, 769, 3071, 3072, 3073])
@pytest.mark.parametrize("n", [8193, 22529])
def test_leading_missing_block(n, lead):
    check(columns(n, 17, lead, 3, seed=lead))
