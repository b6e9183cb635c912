"""Exact pair counts of ICI-Kendall-tau from sign-vector products: a reference that shares nothing with the pair
kernel, cheap enough to check every pair of a run with billions of them at small n.

A column x of n rows gets ranks r (rows missing in x rank below every value and tie with each other).  For every
pair of rows a < b (K = n (n - 1) / 2 of them) it has the features

    s_ab = sign(r_b - r_a),   z_ab = [r_a == r_b].

For a column pair (x, y) in the global perspective (all n rows enter):

    S    = sum sx sy = concordant - discordant        ntie = sum zx zy
    xtie = sum zx,  ytie = sum zy,  tot = K,           dis = (tot - xtie - ytie + ntie - S) / 2

so the counts of all pairs at once are two matrix products.  The local perspective drops the B rows missing in both
columns.  Such a row ties, in x, with exactly the rows missing in x, and lies below every other row; so against a row
present in both columns it is concordant, and against any other row it is tied in x or in y.  With Mx, My the rows
missing in x, in y, and Q = n - Mx - My + B the rows present in both:

    S_l    = S - B Q                        ntie_l = ntie - C(B, 2)
    xtie_l = xtie - C(B, 2) - B (Mx - B)     ytie_l = ytie - C(B, 2) - B (My - B)
    tot_l  = C(n - B, 2)

Every sum is an integer below 2^53, so float64 products are exact in any summation order.  raw and taumax follow from
the counts with the pair epilogue's formulas and operation order (icikt_common.cuh, tau_from_counts), elementwise in
float64, so they agree with the kernel bit for bit.

The same code runs on NumPy arrays (CPU, NumpyOps) and on torch tensors of any device (TorchOps)."""
from __future__ import annotations

import math

import numpy as np

COUNT_NAMES = ("dis", "ntie", "xtie", "ytie", "tot", "n_entry", "b")


def ranks(x):
    """(C, n) int32 dense ranks of the columns of x (n, C), NaN = missing: 0 is the lowest group, which holds the
    missing rows when a column has any"""
    x = np.asarray(x, dtype=np.float64)
    v = np.where(np.isnan(x), -np.inf, x).T  # (C, n)
    order = np.argsort(v, axis=1, kind="stable")
    sv = np.take_along_axis(v, order, axis=1)
    new = np.concatenate([np.zeros((v.shape[0], 1), dtype=np.int32),
                          (sv[:, 1:] != sv[:, :-1]).astype(np.int32)], axis=1)
    dense = np.cumsum(new, axis=1, dtype=np.int32)
    r = np.empty_like(dense)
    np.put_along_axis(r, order, dense, axis=1)
    return r


class TorchOps:
    """the few array operations the reference needs, on torch tensors of one device"""

    def __init__(self, torch, device):
        self.t, self.device = torch, device

    def asarray(self, a, dtype=None):
        return self.t.as_tensor(np.ascontiguousarray(a), device=self.device, dtype=getattr(self.t, dtype or "float64"))

    def matmul(self, a, b):
        return a @ b.T

    def sqrt(self, a):
        return self.t.sqrt(a)

    def where(self, c, a, b):
        return self.t.where(c, a, b)

    def full_like(self, a, v):
        return self.t.full_like(a, v)

    def to_numpy(self, a):
        return a.cpu().numpy()


class NumpyOps:
    def asarray(self, a, dtype=None):
        return np.ascontiguousarray(a, dtype=getattr(np, dtype or "float64"))

    def matmul(self, a, b):
        return a @ b.T

    sqrt = staticmethod(np.sqrt)
    where = staticmethod(np.where)

    def full_like(self, a, v):
        return np.full_like(a, v)

    def to_numpy(self, a):
        return np.asarray(a)


class Features:
    """The sign and tie features of the columns of x (n, C; NaN = missing) and their per-column statistics, as
    float64 arrays of `ops` (NumpyOps() or TorchOps(torch, device))."""

    def __init__(self, x, ops=None):
        self.ops = ops or NumpyOps()
        r = ranks(x)
        self.C, self.n = r.shape
        a, b = np.triu_indices(self.n, 1)
        d = r[:, b] - r[:, a]
        self.s = self.ops.asarray(np.sign(d).astype(np.float64))
        self.z = self.ops.asarray((d == 0).astype(np.float64))
        miss = np.isnan(np.asarray(x, dtype=np.float64)).T
        self.m = self.ops.asarray(miss.astype(np.float64))
        self.n_miss = self.ops.asarray(miss.sum(axis=1).astype(np.float64))
        self.tie = self.ops.asarray((d == 0).sum(axis=1).astype(np.float64))
        # distinct values of the column over all rows, the missing group counted as one
        self.groups = self.ops.asarray((r.max(axis=1) + 1).astype(np.float64))

    def take(self, cols):
        """the features of the columns `cols` (an index array or a slice), as a view-like object"""
        out = Features.__new__(Features)
        out.ops, out.n = self.ops, self.n
        for k in ("s", "z", "m", "n_miss", "tie", "groups"):
            setattr(out, k, getattr(self, k)[cols])
        out.C = out.s.shape[0]
        return out


def _pair_stats(X, Y, S, ntie, B, perspective, elementwise):
    """the counts, status, raw and taumax of the pairs of X's and Y's columns from their products (S, ntie, B), as
    matrices (X.C, Y.C), or as vectors for X and Y of equal length when `elementwise`"""
    ops = X.ops
    n = float(X.n)
    with np.errstate(invalid="ignore", divide="ignore"):  # degenerate pairs divide by zero; they are masked below
        return _pair_stats_impl(ops, n, X, Y, S, ntie, B, perspective, elementwise)


def _pair_stats_impl(ops, n, X, Y, S, ntie, B, perspective, elementwise):
    if elementwise:
        Mx, My, xt, yt, gx, gy = X.n_miss, Y.n_miss, X.tie, Y.tie, X.groups, Y.groups
    else:
        Mx, My, xt, yt = X.n_miss[:, None], Y.n_miss[None, :], X.tie[:, None], Y.tie[None, :]
        gx, gy = X.groups[:, None], Y.groups[None, :]
    K = n * (n - 1) / 2
    if perspective == "local":
        Q = n - Mx - My + B
        cb = B * (B - 1) / 2
        S = S - B * Q
        ntie = ntie - cb
        xtie = xt - cb - B * (Mx - B)
        ytie = yt - cb - B * (My - B)
        npr = n - B
        tot = npr * (npr - 1) / 2
        kx = gx - ((Mx > 0) & (Mx == B)) * 1.0  # the missing group is gone when every row missing in x left
        ky = gy - ((My > 0) & (My == B)) * 1.0
    else:
        xtie, ytie = xt + 0 * S, yt + 0 * S
        npr = n + 0 * S
        tot = K + 0 * S
        kx, ky = gx + 0 * S, gy + 0 * S
    dis = (tot - xtie - ytie + ntie - S) / 2
    # status as pair_epilogue sets it: 1 a column all missing, 2 fewer than two rows, 3 a column with one value,
    # 4 every row pair tied in a column
    status = ops.full_like(S, 0.0)
    for code, cond in ((4, (xtie == tot) | (ytie == tot)), (3, (kx == 1) | (ky == 1)), (2, npr < 2),
                       (1, (Mx == n) | (My == n))):
        status = ops.where(cond, ops.full_like(S, float(code)), status)
    # tau_from_counts, icikt_common.cuh: the same float64 operations in the same order
    den = ops.sqrt((tot - xtie) * (tot - ytie))
    cmd = tot - xtie - ytie + ntie - 2 * dis
    cpd = tot - xtie - ytie + ntie
    raw = cmd / den
    raw = ops.where(raw > 1, ops.full_like(raw, 1.0), ops.where(raw < -1, ops.full_like(raw, -1.0), raw))
    taumax = cpd / den
    ok = status == 0
    nan = ops.full_like(raw, float("nan"))
    return dict(dis=dis, ntie=ntie, xtie=xtie, ytie=ytie, tot=tot, n_entry=npr, b=B + 0 * S, S=S, status=status,
                raw=ops.where(ok, raw, nan), taumax=ops.where(ok, taumax, nan))


def block(X, Y, perspective="global"):
    """counts, status, raw and taumax of every pair (X's column i, Y's column j) as (X.C, Y.C) float64 matrices"""
    ops = X.ops
    return _pair_stats(X, Y, ops.matmul(X.s, Y.s), ops.matmul(X.z, Y.z), ops.matmul(X.m, Y.m), perspective, False)


def pairs(F, pi, pj, perspective="global"):
    """the same for the listed pairs (F's column pi[k], F's column pj[k]), as vectors"""
    X, Y = F.take(pi), F.take(pj)
    return _pair_stats(X, Y, (X.s * Y.s).sum(1), (X.z * Y.z).sum(1), (X.m * Y.m).sum(1), perspective, True)


def counts_matrix(st, ops=None):
    """(P, 7) int64 counts in COUNT_NAMES order, and int32 status, from the vectors of pairs()"""
    ops = ops or NumpyOps()
    c = np.stack([ops.to_numpy(st[k]) for k in COUNT_NAMES], axis=1)
    assert np.array_equal(c, np.round(c)), "a count is not an integer"
    return c.astype(np.int64), ops.to_numpy(st["status"]).astype(np.int32)


def pair_index(C, p):
    """(i, j) of pair p of the combn order of C columns (then the diagonal), with exact integers"""
    ptri = C * (C - 1) // 2
    if p >= ptri:
        return p - ptri, p - ptri
    b = 2 * C - 1
    i = (b - math.isqrt(b * b - 8 * p)) // 2
    while i > 0 and row_start(C, i) > p:
        i -= 1
    while i + 1 < C - 1 and row_start(C, i + 1) <= p:
        i += 1
    return i, i + 1 + p - row_start(C, i)


def row_start(C, i):
    """the first pair of row i in the combn order"""
    return i * (2 * C - i - 1) // 2
