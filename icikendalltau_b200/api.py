"""Host-side mirror of the reference's R interface for the ICI-Kendall-tau path.

Same function names, argument meaning, result names and error/warning texts as the
reference (paths relative to the reference repository):

  ici_kt                 R/RcppExports.R:62-64 -> src/kendallc.cpp:166-366
  ici_kendalltau         R/kendalltau.R:96-179  (+ setup_comparisons :181-278,
                                                  scale_and_reshape :357-421)
  kt_fast                R/kendalltau.R:448-545 (+ kt_split :310-354)
  pairwise_completeness  R/kendalltau.R:563-629

All pair arithmetic runs in libicikt_b200.so on the GPU (no CPU fallback); this module
only validates arguments, plans the pair list and reshapes the results, which is what
the R host code keeps doing in the reference-side integration (INTEGRATION.md).
R is not available in the build image, so this Python layer is the executable host.
"""
from __future__ import annotations

import logging
import time
import warnings

import numpy as np

from . import _lib

log = logging.getLogger("icikendalltau_b200")

WARN_SINGLE_VALUE = "Warning: The vectors only have a single value, NA returned!"              # src/kendallc.cpp:225
WARN_SINGLE_UNIQUE = "Warning: Either 'X' or 'Y' have only a single unique value, NA returned!"  # :238
WARN_ALL_TIED = "Warning: Ties equal the total, NA returned!"                                   # :292
_STATUS_WARNING = {2: WARN_SINGLE_VALUE, 3: WARN_SINGLE_UNIQUE, 4: WARN_ALL_TIED}


class IciKtResult(dict):
    """Named vector c(tau, pvalue, tau_max, completeness) (src/kendallc.cpp:171-172)."""

    NAMES = ("tau", "pvalue", "tau_max", "completeness")

    def __getitem__(self, k):
        if isinstance(k, int):
            k = self.NAMES[k]
        return dict.__getitem__(self, k)

    def as_array(self):
        return np.array([dict.__getitem__(self, k) for k in self.NAMES])


def _warn_status(status):
    for code, text in _STATUS_WARNING.items():
        cnt = int((status == code).sum())
        if cnt:
            warnings.warn(text if cnt == 1 else f"{text} ({cnt} pairs)", RuntimeWarning, stacklevel=3)


def _warn_status_counts(counts):
    for code, text in _STATUS_WARNING.items():
        cnt = int(counts[code])
        if cnt:
            warnings.warn(text if cnt == 1 else f"{text} ({cnt} pairs)", RuntimeWarning, stacklevel=3)


def _colnames_of(x, colnames, arg):
    """check_if_colnames_null + transform_to_matrix + check_if_numeric (R/utils.R:25-66)."""
    names = colnames
    try:
        import pandas as pd
        if isinstance(x, pd.DataFrame):
            log.info("`%s` is a data.frame, converting to matrix ...", arg)
            names = list(x.columns) if names is None else names
            x = x.to_numpy()
    except ImportError:  # pandas is optional
        pass
    if _lib.is_sparse(x):  # stays sparse: the library takes the stored entries (entries not stored are 0.0)
        if len(x.shape) != 2:
            raise ValueError(f"`{arg}` must be matrix-like (features x samples)")
        if names is None:
            raise ValueError(f"Colnames of `{arg}` must be be specified.")
        names = list(names)
        if len(names) != x.shape[1]:
            raise ValueError(f"`colnames` has {len(names)} entries but `{arg}` has {x.shape[1]} columns")
        if not (np.issubdtype(x.dtype, np.floating) or np.issubdtype(x.dtype, np.integer)):
            raise TypeError(f"`{arg}` must be a numeric type.")
        return _lib.canonical_csc(x), names
    arr = np.asarray(x)
    if arr.ndim != 2:
        raise ValueError(f"`{arg}` must be matrix-like (features x samples)")
    if names is None:
        raise ValueError(f"Colnames of `{arg}` must be be specified.")
    names = list(names)
    if len(names) != arr.shape[1]:
        raise ValueError(f"`colnames` has {len(names)} entries but `{arg}` has {arr.shape[1]} columns")
    if not (np.issubdtype(arr.dtype, np.floating) or np.issubdtype(arr.dtype, np.integer)):
        raise TypeError(f"`{arg}` must be a numeric type.")
    return np.asarray(arr, dtype=np.float64), names


def setup_missing_matrix(data_matrix, global_na):
    """R/utils.R:1-23.  Used for `keep`, `n_good` and the odd corner where global_na has no NA."""
    data = np.asarray(data_matrix, dtype=np.float64)
    excl = np.zeros(data.shape, dtype=bool)
    g = [float(v) for v in global_na]
    if any(np.isnan(v) for v in g):
        excl |= np.isnan(data)
    if any(np.isinf(v) for v in g):
        excl |= np.isinf(data)
    for v in g:
        if np.isfinite(v):
            excl |= (data == v)
    return excl


def _keep_and_n_good(data, global_na):
    """keep (C x n: not missing) and n_good (per column) of setup_missing_matrix (R/utils.R:1-23).  For
    sparse input both come from the stored entries: an entry not stored is 0.0, missing iff global_na holds a 0
    (the same rule setup_missing_matrix applies to it)."""
    if not _lib.is_sparse(data):
        exclude_loc = setup_missing_matrix(data, global_na)
        return (~exclude_loc).T, (~exclude_loc).sum(axis=0)
    m = _lib.CSC(data)
    n, C = m.shape
    implicit_good = not setup_missing_matrix(np.zeros(1), global_na)[0]
    stored_good = ~setup_missing_matrix(m.values, global_na)
    per_col = np.diff(m.colptr)
    col = np.repeat(np.arange(C), per_col)
    n_good = np.bincount(col, weights=stored_good, minlength=C).astype(np.int64)
    if implicit_good:
        n_good += n - per_col
    keep = np.full((C, n), implicit_good, dtype=bool)
    keep[col, m.rowidx] = stored_good
    return keep, n_good


def setup_comparisons(samples, include_only=None, diag_good=True, include_arg="include_only"):
    """R/kendalltau.R:181-247.  Returns (pi, pj, all_pairs) with 0-based indices; all_pairs is
    True when the list is exactly combn order (+ diagonal), so no explicit list is needed."""
    n_sample = len(samples)
    iu = np.triu_indices(n_sample, k=1)
    pi, pj = iu[0].astype(np.int32), iu[1].astype(np.int32)
    if not diag_good:
        d = np.arange(n_sample, dtype=np.int32)
        pi, pj = np.concatenate([pi, d]), np.concatenate([pj, d])
    all_pairs = True
    if include_only is not None:
        all_pairs = False
        index = {}
        for k, s in enumerate(samples):
            index.setdefault(s, k)
        try:
            import pandas as pd
            if isinstance(include_only, pd.DataFrame):
                include_only = [list(include_only.iloc[:, c]) for c in range(include_only.shape[1])]
        except ImportError:
            pass
        if isinstance(include_only, dict):
            include_only = list(include_only.values())
        # a list mixing scalars and vectors, the documented list(g1 = "s1", g2 = c("s2", "s3")) form
        # (R/kendalltau.R:86-91): scalars are vectors of length one and paste0 recycles them
        if isinstance(include_only, (list, tuple)) and \
                any(isinstance(v, (list, tuple, np.ndarray)) for v in include_only):
            include_only = [list(v) if isinstance(v, (list, tuple, np.ndarray)) else [v] for v in include_only]
        is_list_of_vectors = isinstance(include_only, (list, tuple)) and len(include_only) > 0 and \
            all(isinstance(v, (list, tuple, np.ndarray)) for v in include_only)
        if is_list_of_vectors:
            if len(include_only) != 2:
                raise ValueError(f"`{include_arg}` must be a vector, a data.frame with two columns, "
                                 f"or list of two vectors. Currently, `length({include_arg})` returns "
                                 f"{len(include_only)}")
            l1, l2 = list(include_only[0]), list(include_only[1])
            m = max(len(l1), len(l2))  # paste0 recycles the shorter vector
            l1 = [l1[k % len(l1)] for k in range(m)]
            l2 = [l2[k % len(l2)] for k in range(m)]
            want = set()
            for a, b in zip(l1, l2):
                if a in index and b in index:
                    want.add((index[a], index[b]))
                    want.add((index[b], index[a]))
            code = pi.astype(np.int64) * n_sample + pj
            wcode = np.array([a * n_sample + b for a, b in want], dtype=np.int64)
            keep = np.isin(code, wcode)
        else:
            inc = include_only if isinstance(include_only, (list, tuple, np.ndarray)) else [include_only]
            idx = np.array([index[s] for s in inc if s in index], dtype=np.int32)
            keep = np.isin(pi, idx) | np.isin(pj, idx)
        pi, pj = pi[keep], pj[keep]
    if pi.size == 0:
        raise ValueError("No comparisons to do. Check the list of column names in "
                         f"`{include_arg}` vs those in the samples.")
    return pi, pj, all_pairs


def ici_kt(x, y, perspective="local", alternative="two.sided", continuity=False, output="simple",
           device=0):
    """Information-content-informed Kendall-tau of two vectors (missing = NaN).

    Returns the named vector tau, pvalue, tau_max, completeness.  Degenerate inputs return
    NaN in all four with the reference's warning; a length mismatch raises.
    """
    x = np.asarray(x, dtype=np.float64).ravel()
    y = np.asarray(y, dtype=np.float64).ravel()
    if x.size != y.size:
        raise ValueError("'X' and 'Y' are not the same length!")  # src/kendallc.cpp:168-170
    if x.size == 0:
        return IciKtResult(zip(IciKtResult.NAMES, [np.nan] * 4))  # all-NA branch, :193-199
    data = np.column_stack([x, y])
    r = _lib.run_pairs(data, (), pi=[0], pj=[1], perspective=perspective, alternative=alternative,
                       continuity=continuity, device=device)
    _warn_status(r["status"])
    res = IciKtResult(tau=r["raw"][0], pvalue=r["pvalue"][0], tau_max=r["taumax"][0],
                      completeness=r["completeness"][0])
    if output != "simple":
        print("\n".join(f"{k}: {v}" for k, v in res.items()))
    return res


def _edge_mask(cor, pvalue, min_abs_cor, max_pvalue):
    """rows of a long table that pass the filter of ici_kendalltau (a bound of None is no condition)"""
    sel = np.ones(len(cor), dtype=bool)
    if min_abs_cor is not None:
        sel &= np.abs(cor) >= min_abs_cor
    if max_pvalue is not None:
        sel &= pvalue <= max_pvalue
    return sel


def _padj_checks(p_adjust, max_padj, return_matrix):
    """the argument checks of p_adjust / max_padj; True when the long table gets a padj column"""
    if p_adjust is None:
        if max_padj is not None:
            raise ValueError("`max_padj` bounds the adjusted p-value: give `p_adjust` too")
        return False
    _lib.padj_method(p_adjust)
    if return_matrix:
        raise ValueError("`p_adjust` and `max_padj` add a column to the long table: pass return_matrix=False")
    return True


def _reshape(names, pi, pj, cols):
    C = len(names)
    out = {}
    for k, v in cols.items():
        m = np.zeros((C, C))
        m[pi, pj] = v
        m[pj, pi] = v
        out[k] = m
    return out


def ici_kendalltau(data_matrix, global_na=(np.nan, np.inf, 0), perspective="global", scale_max=True,
                   diag_good=True, include_only=None, alternative="two.sided", continuity=False,
                   check_timing=False, return_matrix=True, colnames=None, device=0, n_gpus=1,
                   min_abs_cor=None, max_pvalue=None, max_edges=None, p_adjust=None, max_padj=None):
    """All-pairs ICI-Kendall-tau between the columns (samples) of a features x samples matrix.

    Returns a dict with `cor`, `raw`, `pvalue`, `taumax`, `completeness` (C x C matrices),
    `keep`, `run_time` and `names`; with return_matrix=False a long table `cor` (dict of columns
    s1, s2, raw, pvalue, taumax, completeness, cor) like the reference's data.frame.
    n_gpus > 1 spreads the pair order over that many GPUs of the box (the role of the reference's
    furrr workers), still in one library call.

    min_abs_cor / max_pvalue (return_matrix=False, one GPU) keep only the rows of the long table with
    abs(cor) >= min_abs_cor and pvalue <= max_pvalue (a bound of None is no condition; the diagonal rows of
    diag_good are subject to the same mask).  Over all pairs the selection runs on the device window by window
    (_lib.run_edges), so neither the result nor the device memory grows with the number of pairs; degenerate
    pairs never pass and raise no warning there.  max_edges: raise IciktError (ERR_LIMIT) when more computed
    pairs than that pass.  The filtered table over several GPUs is _lib.run_edges(..., devices=[...]), which
    returns the same rows as one GPU.

    p_adjust (return_matrix=False): one of R's p.adjust methods ("bonferroni", "holm", "hochberg", "BH" or "fdr",
    "BY"; not "hommel").  The long table gains a column padj, bit for bit R's p.adjust(pvalue[s1 != s2], method)
    over the computed pairs of the unfiltered table: every pair, or the include_only pairs, with the diagonal pairs
    that diag_good=False computes.  The diag_good rows the host appends (p = 0) are not part of that family and get
    padj = 0.  max_padj keeps the rows with padj <= max_padj, with the same mask rules as max_pvalue (one GPU).  Over
    all pairs with any bound (min_abs_cor, max_pvalue, max_padj) the adjustment runs on the device window by window
    with the filter (_lib.run_edges(p_adjust=...)); otherwise the table's p-values are adjusted by _lib.p_adjust.
    """
    adjusted = _padj_checks(p_adjust, max_padj, return_matrix)
    filtered = min_abs_cor is not None or max_pvalue is not None or max_padj is not None
    if filtered and return_matrix:
        raise ValueError("`min_abs_cor` and `max_pvalue` select rows of the long table: pass return_matrix=False")
    if filtered and n_gpus > 1:
        raise ValueError("`min_abs_cor` and `max_pvalue` run on one GPU: n_gpus must be 1")
    if max_edges is not None and not filtered:
        raise ValueError("`max_edges` limits a filtered table: give `min_abs_cor` or `max_pvalue` too")
    data, names = _colnames_of(data_matrix, colnames, "data_matrix")
    n, C = data.shape
    log.info("Processing missing values ...")
    global_na = [float(v) for v in global_na]
    keep, n_good = _keep_and_n_good(data, global_na)
    log.info("Figuring out comparisons to do ...")
    if include_only is None and (return_matrix or filtered) and not check_timing:
        # every pair, in the library's own order, straight into matrices or filtered on the device: no pair
        # list on the host
        pi = pj = None
        all_pairs = True
        if C < 2 and diag_good:
            raise ValueError("No comparisons to do. Check the list of column names in "
                             "`include_only` vs those in the samples.")
    else:
        pi, pj, all_pairs = setup_comparisons(names, include_only, diag_good)
        n_todo = pi.size

    kw = dict(perspective=perspective, alternative=alternative, continuity=continuity, device=device)
    if check_timing:  # R/kendalltau.R:141-148, 633-669
        rng = np.random.default_rng()
        sel = rng.choice(n_todo, size=min(5, n_todo), replace=False)
        t0 = time.perf_counter()
        _lib.run_pairs(data, global_na, pi=pi[sel], pj=pj[sel], **kw)
        t_total = time.perf_counter() - t0
        t_each = t_total / sel.size
        t_all = t_each * n_todo
        return dict(which=["n_tested", "n_todo", "time_tested", "time_single", "time_all",
                           "time_across_cores", "time_minutes", "time_hours", "time_days"],
                    value=[sel.size, n_todo, t_total, t_each, t_all, t_all, t_all / 60,
                           t_all / 3600, t_all / 216000])

    log.info("Running correlations ...")
    t1 = time.perf_counter()
    if return_matrix and (n_gpus <= 1 or all_pairs):
        # scale_and_reshape on the device: the five C x C matrices come back filled (:357-421)
        if all_pairs and n_gpus > 1:  # every GPU fills and returns its own block of columns
            r = _lib.run_matrices(data, global_na, scale_max, diag_good, n_good, devices=range(n_gpus), **kw)
        elif all_pairs:
            r = _lib.run_matrices(data, global_na, scale_max, diag_good, n_good, **kw)
        else:
            r = _lib.run_matrices(data, global_na, scale_max, diag_good, n_good, pi=pi, pj=pj, **kw)
        run_time = time.perf_counter() - t1
        _warn_status_counts(r["status_counts"])
        log.info("Generating the output matrix ...")
        out = {k: r[k] for k in _lib.MATRIX_NAMES}
        out["keep"] = keep
        out["run_time"] = run_time
        out["names"] = names
        return out
    if filtered and all_pairs:  # selected on the device, window by window
        pk = dict(p_adjust=p_adjust, max_padj=max_padj) if adjusted else {}
        r = _lib.run_edges(data, global_na, min_abs_cor, max_pvalue, scale_max, max_edges or 0,
                           include_diag=not diag_good, **pk, **kw)
        run_time = time.perf_counter() - t1
        pi, pj = r["i"], r["j"]
        raw, pvalue, taumax, completeness, cor = (r[k] for k in ("raw", "pvalue", "taumax", "completeness", "cor"))
        padj = r.get("padj")
    else:
        if all_pairs and n_gpus > 1:  # one call, the pair order sliced over the GPUs inside the library
            r = _lib.run_pairs(data, global_na, include_diag=not diag_good, devices=range(n_gpus), **kw)
        elif all_pairs:
            r = _lib.run_pairs(data, global_na, include_diag=not diag_good, **kw)
        else:
            r = _lib.run_pairs(data, global_na, pi=pi, pj=pj, **kw)
        run_time = time.perf_counter() - t1
        _warn_status(r["status"])

        log.info("Recombining results ...")
        raw, pvalue, taumax, completeness = r["raw"], r["pvalue"], r["taumax"], r["completeness"]
        if scale_max:  # R/kendalltau.R:368-372: max over the pairs actually computed, na.rm
            cor = raw / r["max_taumax"]
        else:
            cor = raw.copy()
        padj = _lib.p_adjust(pvalue, p_adjust, device=device) if adjusted else None
        if filtered:  # include_only: the pair list exists already, the mask runs here
            sel = _edge_mask(cor, pvalue, min_abs_cor, max_pvalue)
            if max_padj is not None:
                sel &= padj <= max_padj
            if max_edges and int(sel.sum()) > max_edges:
                raise _lib.IciktError(_lib.ERR_LIMIT, f"more than max_edges = {max_edges} pairs pass the filter "
                                                      f"({int(sel.sum())})")
            pi, pj, raw, pvalue, taumax, completeness, cor = (
                v[sel] for v in (pi, pj, raw, pvalue, taumax, completeness, cor))
            if adjusted:
                padj = padj[sel]
    if diag_good:  # R/kendalltau.R:374-386 (appended after scaling, never scaled)
        d = np.arange(C, dtype=np.int32)
        dg = n_good / n_good.max()
        dp, dt, dc = np.zeros(C), np.ones(C), n_good / n
        if filtered:
            sel = _edge_mask(dg, dp, min_abs_cor, max_pvalue)
            if max_padj is not None:
                sel &= 0.0 <= max_padj
            d, dg, dp, dt, dc = d[sel], dg[sel], dp[sel], dt[sel], dc[sel]
        if adjusted:
            padj = np.concatenate([padj, np.zeros(d.size)])
        pi, pj = np.concatenate([pi, d]), np.concatenate([pj, d])
        raw, cor = np.concatenate([raw, dg]), np.concatenate([cor, dg])
        pvalue = np.concatenate([pvalue, dp])
        taumax = np.concatenate([taumax, dt])
        completeness = np.concatenate([completeness, dc])
    if not return_matrix:
        nm = np.asarray(names, dtype=object)
        table = dict(s1=nm[pi], s2=nm[pj], raw=raw, pvalue=pvalue, taumax=taumax, completeness=completeness, cor=cor)
        if adjusted:
            table["padj"] = padj
        return dict(cor=table, run_time=run_time, names=names)
    log.info("Generating the output matrix ...")
    out = _reshape(names, pi, pj, dict(cor=cor, raw=raw, pvalue=pvalue, taumax=taumax,
                                        completeness=completeness))
    out["keep"] = keep
    out["run_time"] = run_time
    out["names"] = names
    return out


def ici_kendalltau_topk(data_matrix, k, by="abs", global_na=(np.nan, np.inf, 0), perspective="global",
                        scale_max=True, alternative="two.sided", continuity=False, colnames=None, device=0, n_gpus=1):
    """Every sample's k most correlated partners (a kNN table), over all pairs of a features x samples matrix.

    The candidates of sample c are the samples d != c whose pair is not degenerate, ranked by abs(raw) (by="abs")
    or raw (by="signed") descending, then by column position; c keeps its first min(k, #candidates), best first.
    The selection runs window by window (_lib.run_topk), so neither the result nor the device memory grows with the
    number of pairs; degenerate pairs raise no warning.  n_gpus > 1 spreads the pair order over GPUs 0..n_gpus-1 of
    the box in one library call (`device` is then not used); the lists are the same as on one GPU.  Values are those of ici_kendalltau for the
    same pair, cor = raw / max(taumax over all pairs) if scale_max else raw.

    Returns a dict of (C, k) arrays `index` (int32, -1 where unused), `neighbors` (column names, None where
    unused), `cor`, `raw`, `pvalue`, `taumax`, `completeness` (NaN where unused), plus `n_neighbors` (C,),
    `max_taumax`, `run_time` and `names`.
    """
    if isinstance(k, (bool, np.bool_)) or not isinstance(k, (int, np.integer)) or not 1 <= k <= _lib.TOPK_MAX:
        raise ValueError(f"`k` must be an integer in [1, {_lib.TOPK_MAX}], got {k!r}")
    if by not in _lib.TOPK_BY:
        raise ValueError(f"`by` must be 'abs' or 'signed', got {by!r}")
    data, names = _colnames_of(data_matrix, colnames, "data_matrix")
    global_na = [float(v) for v in global_na]
    log.info("Running correlations ...")
    t1 = time.perf_counter()
    kw = dict(perspective=perspective, alternative=alternative, continuity=continuity, device=device)
    if n_gpus > 1:
        kw["devices"] = range(n_gpus)
    r = _lib.run_topk(data, global_na, int(k), by, scale_max, **kw)
    run_time = time.perf_counter() - t1
    nm = np.empty(len(names) + 1, dtype=object)  # the last entry, None, is what index -1 picks
    for c, v in enumerate(names):
        nm[c] = v
    out = {key: r[key] for key in ("index", "cor", "raw", "pvalue", "taumax", "completeness", "n_neighbors",
                                   "max_taumax")}
    out["neighbors"] = nm[r["index"]]
    out["run_time"] = run_time
    out["names"] = names
    return out


def _cross_data(x, y, xnames, ynames):
    x, xnames = _colnames_of(x, xnames, "x")
    y, ynames = _colnames_of(y, ynames, "y")
    if x.shape[0] != y.shape[0]:
        raise ValueError(f"`x` has {x.shape[0]} rows and `y` has {y.shape[0]}: both need the same features")
    return x, y, xnames, ynames


def _names_by_index(names):
    """names as an object array with a trailing None, which index -1 picks"""
    nm = np.empty(len(names) + 1, dtype=object)
    for c, v in enumerate(names):
        nm[c] = v
    return nm


def ici_kendalltau_cross(x, y, global_na=(np.nan, np.inf, 0), perspective="global", scale_max=True,
                         alternative="two.sided", continuity=False, return_matrix=True, min_abs_cor=None,
                         max_pvalue=None, max_edges=None, xnames=None, ynames=None, device=0, n_gpus=1,
                         p_adjust=None, max_padj=None):
    """ICI-Kendall-tau of every column (sample) of `x` with every column of `y`, both features x samples with the
    same features: query samples against a reference panel, two batches, two feature sets on the same samples.

    Every value is the one ici_kendalltau computes for that pair of columns side by side, with x's column first;
    cor = raw / max(taumax over the Cx x Cy pairs) if scale_max else raw.  Returns a dict with `cor`, `raw`,
    `pvalue`, `taumax`, `completeness` as (Cx, Cy) arrays (row i: x's column i), `xnames`, `ynames` and `run_time`;
    with return_matrix=False a long table `cor` (dict of columns s1 from x, s2 from y, raw, pvalue, taumax,
    completeness, cor) in x-major order.  The pairs run window by window on the device (_lib.run_cross), so device
    memory does not grow with Cx x Cy.  Each degenerate class warns once.

    min_abs_cor / max_pvalue (return_matrix=False) keep only the rows with abs(cor) >= min_abs_cor and
    pvalue <= max_pvalue, selected on the device (_lib.run_cross_edges) with the rules of ici_kendalltau's filtered
    table; max_edges raises IciktError (ERR_LIMIT) when more pairs pass.  One GPU: n_gpus must be 1.  The same
    results over several GPUs are _lib.run_cross(x, y, devices=[...]) and _lib.run_cross_edges(..., devices=[...]),
    which return bit for bit what one GPU returns.

    p_adjust / max_padj (return_matrix=False) as in ici_kendalltau: the long table gains padj, bit for bit R's
    p.adjust(pvalue, method) over all Cx x Cy pairs; with any bound the adjustment runs on the device with the filter
    (_lib.run_cross_edges(p_adjust=...)), otherwise _lib.p_adjust adjusts the table's p-values.
    """
    if n_gpus != 1:
        raise ValueError("the cross calls run on one GPU: n_gpus must be 1")
    adjusted = _padj_checks(p_adjust, max_padj, return_matrix)
    filtered = min_abs_cor is not None or max_pvalue is not None or max_padj is not None
    if filtered and return_matrix:
        raise ValueError("`min_abs_cor` and `max_pvalue` select rows of the long table: pass return_matrix=False")
    if max_edges is not None and not filtered:
        raise ValueError("`max_edges` limits a filtered table: give `min_abs_cor` or `max_pvalue` too")
    x, y, xnames, ynames = _cross_data(x, y, xnames, ynames)
    cx, cy = x.shape[1], y.shape[1]
    global_na = [float(v) for v in global_na]
    kw = dict(perspective=perspective, alternative=alternative, continuity=continuity, device=device)
    log.info("Running correlations ...")
    t1 = time.perf_counter()
    if filtered:
        pk = dict(p_adjust=p_adjust, max_padj=max_padj) if adjusted else {}
        r = _lib.run_cross_edges(x, y, global_na, min_abs_cor, max_pvalue, scale_max, max_edges or 0, **pk, **kw)
        run_time = time.perf_counter() - t1
        xn, yn = np.asarray(xnames, dtype=object), np.asarray(ynames, dtype=object)
        table = dict(s1=xn[r["i"]], s2=yn[r["j"]], raw=r["raw"], pvalue=r["pvalue"], taumax=r["taumax"],
                     completeness=r["completeness"], cor=r["cor"])
        if adjusted:
            table["padj"] = r["padj"]
        return dict(cor=table, run_time=run_time, xnames=xnames, ynames=ynames)
    r = _lib.run_cross(x, y, global_na, **kw)
    run_time = time.perf_counter() - t1
    _warn_status(r["status"])
    cols = {k: r[k] for k in ("raw", "pvalue", "taumax", "completeness")}
    cols["cor"] = r["raw"] / r["max_taumax"] if scale_max else r["raw"].copy()
    if not return_matrix:
        xn, yn = np.asarray(xnames, dtype=object), np.asarray(ynames, dtype=object)
        table = dict(s1=np.repeat(xn, cy), s2=np.tile(yn, cx))
        table.update((k, cols[k]) for k in ("raw", "pvalue", "taumax", "completeness", "cor"))
        if adjusted:
            table["padj"] = _lib.p_adjust(r["pvalue"], p_adjust, device=device)
        return dict(cor=table, run_time=run_time, xnames=xnames, ynames=ynames)
    out = {k: cols[k].reshape(cx, cy) for k in _lib.MATRIX_NAMES}
    out.update(xnames=xnames, ynames=ynames, run_time=run_time)
    return out


def ici_kendalltau_cross_topk(x, y, k, by="abs", side="x", global_na=(np.nan, np.inf, 0), perspective="global",
                              scale_max=True, alternative="two.sided", continuity=False, xnames=None, ynames=None,
                              device=0, n_gpus=1):
    """Each sample's k most correlated partners in the OTHER matrix (x and y: features x samples, same features).

    side="x": for every column of x, its best columns of y (query against reference); "y": for every column of y,
    its best columns of x; "both": the two lists, e.g. for mutual nearest neighbours between two batches.  Ranking,
    padding and values are those of ici_kendalltau_topk over the Cx x Cy pairs; cor = raw / max(taumax over those
    pairs) if scale_max else raw.  The lists are selected on the device window by window (_lib.run_cross_topk) and
    held there only for the requested sides.  One GPU: n_gpus must be 1.  The same lists over several GPUs are
    _lib.run_cross_topk(x, y, ..., devices=[...]), which returns bit for bit what one GPU returns.

    Returns a dict with key "x" and/or "y": per side the dict ici_kendalltau_topk returns (`index`, `neighbors` --
    names from the other matrix --, `cor`, `raw`, `pvalue`, `taumax`, `completeness`, `n_neighbors`, `max_taumax`,
    `run_time`, and `names`, the side's own column names).
    """
    if isinstance(k, (bool, np.bool_)) or not isinstance(k, (int, np.integer)) or not 1 <= k <= _lib.TOPK_MAX:
        raise ValueError(f"`k` must be an integer in [1, {_lib.TOPK_MAX}], got {k!r}")
    if by not in _lib.TOPK_BY:
        raise ValueError(f"`by` must be 'abs' or 'signed', got {by!r}")
    if side not in _lib.CROSS_SIDES:
        raise ValueError(f"`side` must be 'x', 'y' or 'both', got {side!r}")
    if n_gpus != 1:
        raise ValueError("the cross calls run on one GPU: n_gpus must be 1")
    x, y, xnames, ynames = _cross_data(x, y, xnames, ynames)
    global_na = [float(v) for v in global_na]
    log.info("Running correlations ...")
    t1 = time.perf_counter()
    r = _lib.run_cross_topk(x, y, global_na, int(k), by, scale_max, side, perspective=perspective,
                            alternative=alternative, continuity=continuity, device=device)
    run_time = time.perf_counter() - t1
    out = {}
    for key, own, other in (("x", xnames, ynames), ("y", ynames, xnames)):
        if key + "_side" not in r:
            continue
        lists = r[key + "_side"]
        d = {f: lists[f] for f in ("index", "cor", "raw", "pvalue", "taumax", "completeness", "n_neighbors")}
        d["neighbors"] = _names_by_index(other)[lists["index"]]
        d.update(max_taumax=r["max_taumax"], run_time=run_time, names=own)
        out[key] = d
    return out


_NA_METHODS = ("all.obs", "complete.obs", "pairwise.complete.obs", "everything", "na.or.complete")


def _match_arg(use):
    hits = [m for m in _NA_METHODS if m.startswith(use)]
    if use in _NA_METHODS:
        return use
    if len(hits) != 1:
        raise ValueError("'arg' should be one of " + ", ".join(f"'{m}'" for m in _NA_METHODS))
    return hits[0]


def kt_fast(x, y=None, use="everything", alternative="two.sided", continuity=False,
            return_matrix=True, colnames=None, device=0):
    """Plain Kendall-tau-b through the ICI kernel (R/kendalltau.R:448-545).

    As in the reference, `alternative` and `continuity` are accepted but not forwarded to the
    pair kernel (kt_split calls ici_kt(tmp_x, tmp_y) with defaults, :341), and the (i,i) pairs
    are computed (diag_good = FALSE, :479).
    """
    na_method = _match_arg(use)
    if na_method == "na.or.complete":
        raise ValueError("'na.or.complete' is not a supported value for `use`. Please use one of "
                         "all.obs complete.obs pairwise.complete everthing.")
    xa = np.asarray(x) if not hasattr(x, "columns") else None
    if y is None:
        if xa is not None and xa.ndim < 2:
            raise ValueError("`x` and `y` should both be provided as vectors, or `x` should be "
                             "matrix-like. `x` is a single vector, and `y` is `NULL`.")
        data, names = _colnames_of(x, colnames, "x")
    else:
        ya = np.asarray(y)
        if (xa is None or xa.ndim > 1) or ya.ndim > 1:
            raise ValueError("Both `x` and `y` must be vectors.")
        data = np.column_stack([np.asarray(x, dtype=np.float64), np.asarray(y, dtype=np.float64)])
        names = list(colnames) if colnames is not None else ["x", "y"]
    n, C = data.shape
    na_vals = np.isnan(data)
    any_na = bool(na_vals.any())
    no_na_rows = na_vals.sum(axis=1) == 0
    pi, pj, _ = setup_comparisons(names, None, diag_good=False)
    P = pi.size
    do = True
    if na_method in ("everything", "all.obs") and any_na:
        do = False
    if na_method == "complete.obs":  # :491 (the reference misspells the pairwise alternative)
        if no_na_rows.sum() == 0:
            do = False
        else:
            data = data[no_na_rows, :]
    tau = np.full(P, np.nan)
    pv = np.full(P, np.nan)
    t1 = time.perf_counter()
    if do:
        kw = dict(perspective="local", alternative="two.sided", continuity=False, device=device)
        if na_method == "pairwise.complete.obs" and np.isnan(data).any():
            # Rows with a missing value in either column are dropped per pair (:323-331).  The pair
            # kernel does that on the device (complete-observations mode); only pairs it flags as
            # unsupported (a column whose missing rows tie with its minimum in fp64) are filtered
            # here and run as two-column problems.
            r = _lib.run_pairs(data, (), include_diag=True, **dict(kw, perspective="complete"))
            tau, pv = r["raw"].copy(), r["pvalue"].copy()
            redo = np.nonzero(r["status"] == 9)[0]
            r["status"][redo] = 0
            _warn_status(r["status"])
            for k in redo:
                good = ~np.isnan(data[:, pi[k]]) & ~np.isnan(data[:, pj[k]])
                tau[k] = pv[k] = np.nan
                if good.sum() == 0:
                    continue
                sub = np.column_stack([data[good, pi[k]], data[good, pj[k]]])
                r2 = _lib.run_pairs(sub, (), pi=[0], pj=[1], **kw)
                _warn_status(r2["status"])
                tau[k], pv[k] = r2["raw"][0], r2["pvalue"][0]
        else:
            r = _lib.run_pairs(data, (), include_diag=True, **kw)
            _warn_status(r["status"])
            tau, pv = r["raw"], r["pvalue"]
    run_time = time.perf_counter() - t1 if do else 0.0
    if not return_matrix:
        nm = np.asarray(names, dtype=object)
        return dict(tau=dict(s1=nm[pi], s2=nm[pj], tau=tau, pvalue=pv), run_time=run_time, names=names)
    out = _reshape(names, pi, pj, dict(tau=tau, pvalue=pv))
    out["run_time"] = run_time
    out["names"] = names
    return out


def pairwise_completeness(data_matrix, global_na=(np.nan, np.inf, 0), include_only=None,
                          return_matrix=True, colnames=None, device=0):
    """1 - (rows missing in either sample) / n for every pair incl. (i,i) (R/kendalltau.R:563-629).

    A by-product of the pair kernel's missing-row masks: the global-perspective completeness of
    the ICI path is exactly this quantity (tests/testthat/test-kendall-tau.R:138-151).
    """
    data, names = _colnames_of(data_matrix, colnames, "data_matrix")
    n, C = data.shape
    global_na = [float(v) for v in global_na]
    # missing-row bit masks and popc(x | y) on the device; no pair kernel runs
    if include_only is None and return_matrix:  # the pair order itself is not needed
        return _lib.pairwise_completeness(data, global_na, want_matrix=True, want_pairs=False, device=device)["matrix"]
    pi, pj, all_pairs = setup_comparisons(names, include_only, diag_good=False)
    if all_pairs:
        r = _lib.pairwise_completeness(data, global_na, device=device)
    else:
        r = _lib.pairwise_completeness(data, global_na, pi=pi, pj=pj, device=device)
    missing, comp = r["missing"].astype(np.float64), r["completeness"]
    if not return_matrix:
        nm = np.asarray(names, dtype=object)
        return dict(s1=nm[pi], s2=nm[pj], missingness=missing, completeness=comp)
    return _reshape(names, pi, pj, dict(completeness=comp))["completeness"]
