"""The identity that lets pass A leave the other column's lowest-rank (zero) keys out (DESIGN.md section 2),
on a one-bit wavelet-matrix model of the pass: for the sequence seq pass A sees (x's first group emitted in ascending
order, then the gathered keys) and seq' = seq without its zero keys,
    INV(seq) = PassA(seq' + padding) - cconst + sum over zero keys of #(nonzero keys before it),
where cconst, the raw count of y's own sorted keys, is the same with or without y's zeros.  Random and
adversarial sequences: all keys zero, no zeros, zeros only in x's first group, zeros only after it, and
lengths on either side of a thread-range boundary."""
import numpy as np
import pytest


def raw(keys, L):
    """pass A's raw count: per bit from the top, the ones before every zero, then a stable partition"""
    s, tot = list(keys), 0
    for b in range(L - 1, -1, -1):
        ones = 0
        for v in s:
            if (v >> b) & 1:
                ones += 1
            else:
                tot += ones
        s = [v for v in s if not (v >> b) & 1] + [v for v in s if (v >> b) & 1]
    return tot


def inversions(keys):
    a = np.asarray(keys)
    return int(sum(int((a[:i] > a[i]).sum()) for i in range(len(a))))


def compacted(first, gathered):
    """seq' as a compacting gather writes it and the zero term: the first group's nonzero keys, then the
    gathered nonzero keys; a gathered zero key adds its write position (nonzero keys already written)"""
    seq = [v for v in first if v]
    zt = 0
    for v in gathered:
        if v:
            seq.append(v)
        else:
            zt += len(seq)
    return seq, zt


def check(first, gathered, L, R):
    first = sorted(first)  # x's first group is emitted in ascending y order
    seq = first + list(gathered)
    ys = sorted(seq)
    cap = -(-max(len(seq), 1) // R) * R
    pad = (1 << L) - 1
    cconst = raw(ys + [pad] * (cap - len(ys)), L)
    assert raw([v for v in ys if v] + [pad] * (cap - len(ys)), L) == cconst
    full = raw(seq + [pad] * (cap - len(seq)), L) - cconst
    sq, zt = compacted(first, gathered)
    # the compacted sequence is padded up to the same capacity: threads past len' only see padding
    comp = raw(sq + [pad] * (cap - len(sq)), L) - cconst + zt
    assert full == inversions(seq) == comp
    # closed form: sum of gathered zero positions q_z (in seq) - m' b' - m'(m'-1)/2
    b1 = sum(1 for v in first if v == 0)
    qz = [len(first) + i for i, v in enumerate(gathered) if v == 0]
    m1 = len(qz)
    assert zt == sum(qz) - m1 * b1 - m1 * (m1 - 1) // 2


def split(rng, keys):
    f = int(rng.integers(0, len(keys) + 1))
    return list(keys[:f]), list(keys[f:])


@pytest.mark.parametrize("seed", range(60))
def test_random_sequences(seed):
    rng = np.random.default_rng(seed)
    n = int(rng.integers(2, 150))
    K = int(rng.integers(2, 60))
    L = max(1, int(np.ceil(np.log2(K))))
    y = rng.integers(0, K, n)
    y[rng.random(n) < rng.random()] = 0
    first, gathered = split(rng, rng.permutation(y))
    check(first, gathered, L, R=8 * int(rng.choice([1, 3, 5])))


def test_adversarial_sequences():
    rng = np.random.default_rng(7)
    for L in (1, 2, 3, 5, 6):
        K = 1 << L
        for n in (1, 2, 9, 40, 97):
            nz = rng.integers(1, K, n)
            check([0] * 3, [0] * n, L, R=8)                            # all keys zero
            check(list(nz[: n // 3]), list(nz[n // 3:]), L, R=8)       # no zeros
            check([0] * 5 + list(nz[:2]), list(nz[2:]), L, R=8)        # zeros only in the first group
            g = list(nz)
            for i in rng.choice(n, size=max(1, n // 4), replace=False):
                g[i] = 0
            check(list(nz[:3]), g, L, R=8)                             # zeros only after it
            check([], g, L, R=8)


@pytest.mark.parametrize("R", [8, 24, 40])
def test_lengths_around_a_range_boundary(R):
    """len' = k R - 1, k R, k R + 1: the thread that straddles len' pads its own range, later ones idle"""
    rng = np.random.default_rng(R)
    L = 5
    for k in (1, 2, 3):
        for d in (-1, 0, 1):
            ln = k * R + d
            nz = list(rng.integers(1, 1 << L, ln))
            zeros = int(rng.integers(1, 2 * R))
            g = nz + [0] * zeros
            g = [g[i] for i in rng.permutation(len(g))]
            check([0, 0] + nz[:1], g, L, R)
