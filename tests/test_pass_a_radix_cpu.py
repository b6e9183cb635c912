"""Pass A's two level structures (DESIGN.md section 2) on a model of count_pass: two-bit levels above bit 4 and
the count-only low-nibble level, or with radix-16 levels (the nibble tree's count plus a stable partition by the
4-bit digit) on the bits from 4 up to the highest multiple of 4 below L.  Under both,
    raw(seq) - raw(sorted seq) = INV(seq)
for every L from 1 to 16, with leading zero blocks, tail padding (2^L - 1) and ties, although raw(sorted seq), the
column constant cconst, differs between the structures.  The host picks the structure from n alone; wherever it
picks radix levels, every tier and the complete-observations mode run the two-buffer kernel in shared memory."""
import numpy as np
import pytest

from icikendalltau_b200 import _lib


def levels(L, radix):
    """count_pass's levels from the top: ('two', s) on bits s+1, s; ('radix', s) and the final ('nibble', 0)"""
    nr = (L - 4) >> 2 if radix and L > 4 else 0
    out = [("two", s) for s in range((L - 1) & ~1, 3 + 4 * nr, -2)]
    out += [("radix", s) for s in range(4 * nr, 3, -4)]
    return out + [("nibble", 0)]


def two_bit(seq, s):
    hi = [(v >> (s + 1)) & 1 for v in seq]
    tot = ones = 0
    for h in hi:  # bit s+1 in the level's order
        ones += h
        tot += 0 if h else ones
    part = [v for v in seq if not (v >> (s + 1)) & 1] + [v for v in seq if (v >> (s + 1)) & 1]
    ones = 0
    for v in part:  # bit s after the partition by bit s+1
        if (v >> s) & 1:
            ones += 1
        else:
            tot += ones
    return tot, sorted(seq, key=lambda v: (v >> s) & 3)  # stable


def tree(seq, s):
    """the nibble tree at bit s: per key and bit k of its digit that is 0, the earlier keys agreeing with it on
    the digit's bits above k that have bit k set"""
    tot = 0
    for k in range(4):
        seen = {}
        for v in seq:
            d = (v >> s) & 15
            node = d >> (k + 1)
            if (d >> k) & 1:
                seen[node] = seen.get(node, 0) + 1
            else:
                tot += seen.get(node, 0)
    return tot


def raw(seq, L, radix):
    tot, s_ = 0, list(seq)
    for kind, s in levels(L, radix):
        if kind == "two":
            c, s_ = two_bit(s_, s)
        else:
            c = tree(s_, s)
            s_ = sorted(s_, key=lambda v: (v >> s) & 15)
        tot += c
    return tot


def inversions(seq):
    a = np.asarray(seq)
    return int(sum(int((a[:i] > a[i]).sum()) for i in range(len(a))))


@pytest.mark.parametrize("L", range(1, 17))
def test_identity_under_both_structures(L):
    rng = np.random.default_rng(L)
    for trial in range(6):
        n = int(rng.integers(1, 120))
        K = int(rng.integers(1, min(n, 1 << L) + 1))  # ties when K < n
        vals = np.sort(rng.choice(1 << L, size=K, replace=False)) if K < (1 << L) else np.arange(1 << L)
        seq = [int(v) for v in rng.choice(vals, size=n)]
        lead = int(rng.integers(0, 20)) if trial % 2 else 0
        pad = int(rng.integers(0, 20)) if trial % 3 else 0
        seq = [0] * lead + seq + [(1 << L) - 1] * pad
        for radix in (False, True):
            assert raw(seq, L, radix) - raw(sorted(seq), L, radix) == inversions(seq), (L, radix, seq)
    assert levels(L, True) != levels(L, False) or L < 8


def test_constants_differ_between_structures():
    rng = np.random.default_rng(9)
    y = sorted(int(v) for v in rng.integers(0, 1 << 9, size=300))
    assert raw(y, 9, False) != raw(y, 9, True)


def test_host_choice_agrees_with_the_launch_shapes():
    chosen = [n for n in range(1, 65536) if _lib.pass_a_radix(n)]
    assert chosen == list(range(chosen[0], chosen[-1] + 1)) and chosen[0] == 8193  # above the fused column kernel
    for n in range(chosen[0], chosen[-1] + 1, 7):
        for tier in (0, 1, 2):
            assert _lib.launch_shape(n, tier)["variant"] == "smem", (n, tier)
        assert _lib.launch_shape(n, 0, complete_obs=True)["variant"] == "smem", n
    assert _lib.pass_a_radix(20000) and not _lib.pass_a_radix(60000)  # the target / config 4
