"""Synthetic workloads of BASELINE.json (SURVEY.md 8d).  Seeds are fixed: 1000 + config number.

Left-censored configs: feature mean mu_f ~ N(10, 2), value exp(mu_f + N(0, 0.5)) (fp64,
tie-free), then every entry below the GLOBAL quantile q becomes NaN -- missingness is
correlated across samples like a real limit of detection.  Config 4 is count data
(negative binomial, zeros missing) with heavy ties.
"""
from __future__ import annotations

import numpy as np

WORKLOADS = {
    # name: (n_features, n_samples, censor quantile, perspective, kind)
    "config1": (6887, 96, 0.0, "global", "yeast"),  # the bundled data set, zeros missing (tests/golden)
    "config2": (5000, 100, 0.20, "global", "lognormal"),
    "config3": (20000, 1000, 0.25, "local", "lognormal"),
    "config4": (60000, 200, 0.0, "global", "counts"),
    "config5": (2000, 5000, 0.20, "global", "lognormal"),
    "target": (20000, 2000, 0.25, "global", "lognormal"),
}
SEEDS = {"config1": 1001, "config2": 1002, "config3": 1003, "config4": 1004, "config5": 1005, "target": 1006}


def left_censored(n, C, q, seed):
    rng = np.random.default_rng(seed)
    mu = rng.normal(10.0, 2.0, size=(n, 1))
    x = np.exp(mu + rng.normal(0.0, 0.5, size=(n, C)))
    if q > 0:
        thr = np.quantile(x, q)
        x[x < thr] = np.nan
    return np.asfortranarray(x)


def count_matrix(n, C, seed, min_present=14000):
    rng = np.random.default_rng(seed)
    mu = np.exp(rng.normal(1.0, 2.5, size=(n, 1)))
    depth = rng.uniform(0.5, 2.0, size=(1, C))
    mean = mu * depth
    size = 2.0
    lam = rng.gamma(shape=size, scale=mean / size)
    x = rng.poisson(lam).astype(np.float64)
    # keep every column's missing group inside the reference's int32 domain (SURVEY.md 8a)
    for c in range(C):
        short = min_present - int((x[:, c] > 0).sum())
        if short > 0:
            z = np.nonzero(x[:, c] == 0)[0]
            x[rng.choice(z, size=short, replace=False), c] = 1.0
    x[x == 0] = np.nan
    return np.asfortranarray(x)


def make(name, n=None, C=None, seed=None):
    """Returns (matrix with NaN = missing, perspective)."""
    n0, C0, q, persp, kind = WORKLOADS[name]
    n, C = n or n0, C or C0
    seed = SEEDS[name] if seed is None else seed
    if kind == "yeast":
        # BASELINE config 1: the reference's bundled yeast RNA-seq counts (6 887 x 96), zeros -> missing
        # as ici_kendalltau's default global_na does; fixture made by tests/golden/make_golden.py (stored as
        # per-column ranks, which give the pair results of the original values)
        import os
        here = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
        x = np.array(np.load(os.path.join(here, "tests", "golden", "yeast_missing.npz"))["data"], dtype=np.float64)
        x[x == 0] = np.nan
        return np.asfortranarray(x[:n, :C]), persp
    if kind == "counts":
        return count_matrix(n, C, seed, min_present=min(14000, max(2, n // 4))), persp
    return left_censored(n, C, q, seed), persp
