"""R's stats::p.adjust for bonferroni, holm, hochberg, BH (fdr) and BY, restated line by line in NumPy.

    p.adjust <- function(p, method, n = length(p)) {
        nna <- !is.na(p); p <- p[nna]          # n is evaluated lazily: after the drop, n = m
        lp <- length(p)
        if (n <= 1) return(p0)
        bonferroni = pmin(1, n * p)
        holm     = { i <- seq_len(lp); o <- order(p);                 pmin(1, cummax((n + 1L - i) * p[o]))[ro] }
        hochberg = { i <- lp:1L; o <- order(p, decreasing = TRUE);   pmin(1, cummin((n + 1L - i) * p[o]))[ro] }
        BH       = { i <- lp:1L; o <- order(p, decreasing = TRUE);   pmin(1, cummin(n / i * p[o]))[ro] }
        BY       = { i <- lp:1L; o <- order(p, decreasing = TRUE); q <- sum(1 / (1L:n))
                     pmin(1, cummin(q * n / i * p[o]))[ro] }

Every operation is the same IEEE double operation in the same order; BY's q is R's sum, which accumulates the double
terms 1/k in a long double (np.longdouble: the 80-bit x87 format on x86-64) and rounds once.  Hommel is not here.
"""
from __future__ import annotations

import numpy as np

METHODS = ("bonferroni", "holm", "hochberg", "BH", "BY")


def by_q(m, chunk=1 << 22):
    """sum(1/(1:m)) as R computes it: double terms, a sequential long double sum, one rounding to double"""
    s = np.longdouble(0)
    for lo in range(1, m + 1, chunk):
        t = (1.0 / np.arange(lo, min(m + 1, lo + chunk), dtype=np.float64)).astype(np.longdouble)
        t[0] += s  # the running sum enters the chunk's first addition: the same additions in the same order
        s = np.add.accumulate(t)[-1]
    return float(s)


def p_adjust(p, method):
    """R's p.adjust(p, method) on a float64 array; NaN entries stay as they are"""
    if method == "fdr":
        method = "BH"
    if method not in METHODS:
        raise ValueError(f"method must be one of {METHODS}")
    p0 = np.array(p, dtype=np.float64, copy=True)
    nna = ~np.isnan(p0)
    x = p0[nna]
    n = x.size
    if n <= 1:
        return p0
    if method == "bonferroni":
        adj = np.minimum(1.0, np.float64(n) * x)
    elif method == "holm":
        i = np.arange(1, n + 1, dtype=np.float64)
        o = np.argsort(x, kind="stable")
        v = (np.float64(n + 1) - i) * x[o]
        adj = np.empty(n)
        adj[o] = np.minimum(1.0, np.maximum.accumulate(v))
    else:
        i = np.arange(n, 0, -1, dtype=np.float64)  # lp:1L
        o = np.argsort(-x, kind="stable")  # decreasing
        if method == "hochberg":
            v = (np.float64(n + 1) - i) * x[o]
        elif method == "BH":
            v = (np.float64(n) / i) * x[o]
        else:
            v = ((np.float64(by_q(n)) * np.float64(n)) / i) * x[o]
        adj = np.empty(n)
        adj[o] = np.minimum(1.0, np.minimum.accumulate(v))
    p0[nna] = adj
    return p0
