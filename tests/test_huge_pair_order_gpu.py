"""Pair orders past 2^31 and 2^32 pairs, checked against the sign-vector reference (tests/sign_reference.py) for every
pair, not a sample.

At n = 40 rows the exact integer counts of every pair come from float64 matrix products on the GPU (torch), a method
that shares nothing with the pair kernel; raw and taumax follow with the epilogue's operations, so they are compared
bit for bit.  p-values and completeness of the rows a call returns are compared with the CPU oracle.

  * slices of the per-pair calls straddling 2^31 - 1, 2^31, 2^32, a row start, the last pair and the first diagonal
    pair of a 92 700-column order (4.3e9 pairs), and of a 70 000 x 70 000 cross order (4.9e9 pairs);
  * full windowed walks over 65 600 columns (2 151 647 200 pairs, 2^31 + 4 163 552): filtered edges, p-values
    adjusted over every pair, top-k lists, on tie-free complete data (D1) and on data with ties and left-censored
    missing values (D2), on one device and through several;
  * a 40 000 x 53 700 cross walk (2^31 + 516 352 pairs);
  * every pair of a 6 000-column run with ties and missing values, all seven counts.

Wall times of the walks and of the reference go to $ICIKT_TIMINGS_OUT (a JSON file) when that is set."""
import json
import math
import os
import time

import numpy as np
import pytest

import icikendalltau_b200 as ik
from icikendalltau_b200 import _lib
from oracle import oracle as O
from tests import sign_reference as SR

pytestmark = pytest.mark.gpu

N = 40
K = N * (N - 1) // 2
W = 1 << 26  # the default window of the filtered calls (ICIKT_EDGE_WINDOW)
C_WALK = 65600
P_WALK = C_WALK * (C_WALK - 1) // 2
P_TOL = 1e-12
TIMINGS = {}


def _timed(name, f, *a, **kw):
    t0 = time.perf_counter()
    out = f(*a, **kw)
    TIMINGS[name] = round(time.perf_counter() - t0, 3)
    return out


@pytest.fixture(scope="module", autouse=True)
def _timings_file():
    yield
    path = os.environ.get("ICIKT_TIMINGS_OUT")
    if path and TIMINGS:
        with open(path, "w") as f:
            json.dump(TIMINGS, f, indent=1)


@pytest.fixture(scope="module")
def torch_ops():
    torch = pytest.importorskip("torch")
    if not torch.cuda.is_available():
        pytest.skip("the sign reference runs on the GPU through torch")
    return SR.TorchOps(torch, torch.device("cuda:0"))


def _release(torch_ops):
    _lib.release_workspace()
    torch_ops.t.cuda.empty_cache()


# ---------------------------------------------------------------- data
def _perm_columns(rng, n, C):
    """columns that are random permutations of 0..n-1: complete and tie-free"""
    return np.asfortranarray(np.argsort(rng.random((n, C)), axis=0).astype(np.float64))


def _plant(x, rng, pairs):
    """make column j a noisy copy of column i (a few adjacent ranks swapped) for the pairs (i, j) whose columns are
    not part of an earlier plant, so that every planted pair keeps its strong correlation"""
    src, dst, done = set(), set(), []
    for i, j in pairs:
        if i in dst or j in dst or j in src:
            continue
        y = x[:, i].copy()
        for v in rng.integers(0, x.shape[0] - 1, int(rng.integers(1, 30))):
            a, b = y == v, y == v + 1
            y[a], y[b] = v + 1, v
        x[:, j] = y
        src.add(i)
        dst.add(j)
        done.append((i, j))
    return done


def _walk_plants(C, P):
    """pair indices to plant: just below, at and above 2^31 (the first pair of window 32), around the row start that
    follows, the slices of two and three devices, and the start and end of the last window"""
    i31 = SR.pair_index(C, 2 ** 31)[0]
    rs = SR.row_start(C, i31 + 1)
    last_w = (P - 1) // W * W
    ps = list(range(2 ** 31 - 40, 2 ** 31 + 40)) + list(range(rs - 10, rs + 10))
    ps += list(range(last_w - 10, last_w + 10)) + list(range(P - 40, P))
    for d in (2, 3):
        for k in range(1, d):
            ps += list(range(P * k // d - 5, P * k // d + 5))
    return [SR.pair_index(C, p) for p in ps]


@pytest.fixture(scope="module")
def d1():
    """D1: 65 600 complete tie-free columns with about 200 planted strong pairs"""
    rng = np.random.default_rng(31)
    x = _perm_columns(rng, N, C_WALK)
    planted = _plant(x, rng, _walk_plants(C_WALK, P_WALK))
    assert len(planted) >= 100
    return x, planted


@pytest.fixture(scope="module")
def d2():
    """D2: ties (few distinct values) and left-censored missing values, an all-missing and a constant column"""
    rng = np.random.default_rng(32)
    x = np.round(rng.normal(size=(N, C_WALK)) * 1.3)
    x[x <= -2] = np.nan
    x[:, 7] = np.nan
    x[:, C_WALK - 3] = 1.0
    _plant_ties = _walk_plants(C_WALK, P_WALK)[:120]
    for i, j in _plant_ties:  # strong pairs near 2^31: j copies i with a few values changed
        if j != 7 and i != 7 and j != C_WALK - 3:
            y = x[:, i].copy()
            y[rng.integers(0, N, 3)] = np.round(rng.normal(size=3))
            x[:, j] = y
    return np.asfortranarray(x)


# ---------------------------------------------------------------- reference walk
def reference_walk(F, persp, G=None, M=None, scale_max=True, t_cor=None, topk=(), R=1024):
    """One pass over every pair of F's columns (combn order), or of F x G (cross order), with the sign reference on the
    GPU.  Returns hist (pairs per |S|, status-0 pairs only; exact for complete tie-free data), M (max taumax over
    status-0 pairs), edges (i, j, raw, taumax of the pairs with abs(cor) >= t_cor in pair order; needs M when
    scale_max) and, per `by` in topk (triangle only), the first K_TOP partners of every column by (key desc, partner
    asc) with raw and taumax."""
    torch = F.ops.t
    C = F.C
    cross = G is not None
    Y = G if cross else F
    hist = torch.zeros(K + 1, dtype=torch.int64, device=F.ops.device)
    mx = -math.inf
    edges, lists = [], {by: [] for by in topk}
    jj = torch.arange(Y.C, device=F.ops.device)
    for i0 in range(0, C, R):
        i1 = min(C, i0 + R)
        st = SR.block(F.take(slice(i0, i1)), Y, persp)
        ok = st["status"] == 0
        ii = torch.arange(i0, i1, device=F.ops.device)[:, None]
        tri = ok if cross else ok & (jj[None, :] > ii)
        hist += torch.bincount(st["S"][tri].abs().to(torch.int64), minlength=K + 1)[: K + 1]
        if tri.any():
            mx = max(mx, float(st["taumax"][tri].max()))
        if t_cor is not None:
            cor = st["raw"] / M if scale_max else st["raw"]
            keep = tri & (cor.abs() >= t_cor)
            r, c = torch.nonzero(keep, as_tuple=True)
            edges.append(((r + i0).cpu().numpy(), c.cpu().numpy(), st["raw"][r, c].cpu().numpy(),
                          st["taumax"][r, c].cpu().numpy()))
        for by in topk:
            valid = ok & (jj[None, :] != ii)
            key = st["raw"].abs() if by == "abs" else st["raw"]
            key = torch.where(valid, key, torch.full_like(key, -math.inf))
            vk = torch.topk(key, K_TOP, dim=1).values[:, -1:]
            gt, eq = key > vk, key == vk
            need = K_TOP - gt.sum(1, keepdim=True)
            sel = (gt | (eq & (torch.cumsum(eq.to(torch.int32), 1) <= need))) & valid
            r, c = torch.nonzero(sel, as_tuple=True)
            lists[by].append(((r + i0).cpu().numpy(), c.cpu().numpy(), key[r, c].cpu().numpy(),
                              st["raw"][r, c].cpu().numpy(), st["taumax"][r, c].cpu().numpy()))
        del st
    out = dict(hist=hist.cpu().numpy(), M=mx)
    if t_cor is not None:
        out["edges"] = tuple(np.concatenate([e[k] for e in edges]) for k in range(4)) if edges else None
    for by in topk:
        col, part, key, raw, tm = (np.concatenate([e[k] for e in lists[by]]) for k in range(5))
        o = np.lexsort((part, -key, col))
        col, part, raw, tm = col[o], part[o], raw[o], tm[o]
        r = np.arange(col.size) - np.searchsorted(col, col, side="left")
        assert (r < K_TOP).all()
        idx = np.full((C, K_TOP), -1, dtype=np.int32)
        lr, lt = np.full((C, K_TOP), np.nan), np.full((C, K_TOP), np.nan)
        idx[col, r], lr[col, r], lt[col, r] = part, raw, tm
        out[by] = dict(index=idx, raw=lr, taumax=lt, n_neighbors=np.bincount(col, minlength=C).astype(np.int32))
    return out


K_TOP = 3


def threshold_from_hist(hist, lo=100_000, hi=1_000_000):
    """the smallest |S| whose tail (pairs with |S| >= it) holds at most `hi` pairs; asserts it holds at least `lo`"""
    tail = np.cumsum(hist[::-1])[::-1]
    s = int(np.argmax(tail <= hi))
    assert tail[s] >= lo, f"tail at |S| >= {s}: {tail[s]} pairs"
    return s


# ---------------------------------------------------------------- checks
def bits_equal(a, b):
    """the same doubles bit for bit, NaN (of any payload) where the other is NaN"""
    a, b = np.ascontiguousarray(a, dtype=np.float64), np.ascontiguousarray(b, dtype=np.float64)
    if a.shape != b.shape or not np.array_equal(np.isnan(a), np.isnan(b)):
        return False
    m = ~np.isnan(a)
    return np.array_equal(a[m].view(np.int64), b[m].view(np.int64))


def check_oracle(x, i, j, pvalue, completeness, persp, what):
    """p-values (|dp| <= 1e-12 max(1, z^2) p) and completeness (exact) of pairs (i, j) against the CPU oracle"""
    if i.size == 0:
        return
    ref = O.pair_loop(x, np.minimum(i, j), np.maximum(i, j), perspective=persp, ncore=os.cpu_count() or 1,
                      want_z=True)
    assert bits_equal(completeness, ref["completeness"]), f"{what}: completeness"
    a, b = np.asarray(pvalue), ref["pvalue"]
    assert np.array_equal(a == 0, b == 0), f"{what}: exact-zero p-values"
    nz = b != 0
    err = np.abs(a[nz] - b[nz]) / (np.maximum(1.0, ref["z"][nz] ** 2) * b[nz])
    assert err.size == 0 or err.max() <= P_TOL, f"{what}: p-value error {err.max():.3g}"


def check_edges(got, ref_edges, M, scale_max, what):
    i, j, raw, tm = ref_edges
    assert got["i"].size == i.size, f"{what}: {got['i'].size} rows, reference {i.size}"
    assert np.array_equal(got["i"], i) and np.array_equal(got["j"], j), f"{what}: (i, j)"
    assert bits_equal(got["raw"], raw), f"{what}: raw"
    assert bits_equal(got["taumax"], tm), f"{what}: taumax"
    assert bits_equal(got["cor"], raw / M if scale_max else raw), f"{what}: cor"
    assert bits_equal(got["max_taumax"], M), f"{what}: max_taumax {got['max_taumax']!r} vs {M!r}"


def check_topk(got, ref, M, x, persp, what):
    for name in ("index", "n_neighbors"):
        assert np.array_equal(got[name], ref[name]), f"{what}: {name}"
    assert bits_equal(got["raw"], ref["raw"]) and bits_equal(got["taumax"], ref["taumax"]), f"{what}: raw/taumax"
    assert bits_equal(got["cor"], ref["raw"] / M), f"{what}: cor"
    use = got["index"] >= 0
    c = np.nonzero(use)[0].astype(np.int32)
    check_oracle(x, c, got["index"][use], got["pvalue"][use], got["completeness"][use], persp, what)


# ---------------------------------------------------------------- 1. slices past 2^31 and 2^32
C_SLICE = 92700
P_SLICE = C_SLICE * (C_SLICE - 1) // 2
HALF = 1024


def _slices(C, P):
    i31 = SR.pair_index(C, 2 ** 31)[0]
    out = {"2^31-1": 2 ** 31 - 1, "2^31": 2 ** 31, "2^32": 2 ** 32, "row after 2^31": SR.row_start(C, i31 + 1)}
    out = {k: (v - HALF, v + HALF) for k, v in out.items()}
    out["last pair"] = (P - 2 * HALF, P)
    return out


@pytest.fixture(scope="module")
def slice_data():
    assert P_SLICE > 2 ** 32
    rng = np.random.default_rng(92700)
    x = np.round(rng.normal(size=(N, C_SLICE)) * 2.0)  # ties
    x[x <= -3] = np.nan                                  # left-censored
    return np.asfortranarray(x)


@pytest.mark.parametrize("persp", ["global", "local"])
def test_pair_slices_past_2_32(slice_data, persp, torch_ops):
    x = slice_data
    F = SR.Features(x, torch_ops)
    cases = dict(_slices(C_SLICE, P_SLICE))
    cases["first diagonal pair"] = (P_SLICE - HALF, P_SLICE + HALF)
    for name, (lo, hi) in cases.items():
        diag = hi > P_SLICE
        got = ik.run_pairs(x, (), want_counts=True, perspective=persp, include_diag=diag, pair_lo=lo, pair_hi=hi)
        ij = np.array([SR.pair_index(C_SLICE, p) for p in range(lo, hi)], dtype=np.int32)
        pi, pj = ij[:, 0], ij[:, 1]
        what = f"{persp} {name} [{lo}, {hi})"
        ref = O.pair_loop(x, pi, pj, perspective=persp, ncore=os.cpu_count() or 1, want_counts=True, want_z=True)
        assert np.array_equal(got["status"], ref["status"]), what
        ok = ref["status"] == 0
        assert np.array_equal(got["counts"][ok], ref["counts"][ok]), f"{what}: counts"
        counts, status = SR.counts_matrix(SR.pairs(F, pi, pj, persp), torch_ops)
        assert np.array_equal(status, ref["status"]) and np.array_equal(counts[ok], ref["counts"][ok]), what
        st = SR.pairs(F, pi, pj, persp)
        assert bits_equal(got["raw"], torch_ops.to_numpy(st["raw"])), f"{what}: raw"
        assert bits_equal(got["taumax"], torch_ops.to_numpy(st["taumax"])), f"{what}: taumax"
        assert bits_equal(got["completeness"], ref["completeness"]), f"{what}: completeness"
        check_oracle(x, pi[ok], pj[ok], got["pvalue"][ok], got["completeness"][ok], persp, what)
    _release(torch_ops)


C_CROSS_SLICE = 70000


@pytest.mark.parametrize("devices", [None, [0, 0, 0]])
def test_cross_slices_past_2_32(devices, torch_ops):
    rng = np.random.default_rng(70000)
    x = np.round(rng.normal(size=(N, C_CROSS_SLICE)) * 2.0)
    y = np.round(rng.normal(size=(N, C_CROSS_SLICE)) * 2.0)
    x[x <= -3] = np.nan
    y[y >= 3] = np.nan
    P = C_CROSS_SLICE * C_CROSS_SLICE
    assert P > 2 ** 32
    xy = np.asfortranarray(np.hstack([x, y]))
    F = SR.Features(xy, torch_ops)
    cases = {"2^31-1": 2 ** 31 - 1, "2^31": 2 ** 31, "2^32": 2 ** 32, "row after 2^32": (2 ** 32 // C_CROSS_SLICE + 1) *
             C_CROSS_SLICE}
    cases = {k: (v - HALF, v + HALF) for k, v in cases.items()}
    cases["last pair"] = (P - 2 * HALF, P)
    for name, (lo, hi) in cases.items():
        got = ik.run_cross(x, y, (), devices=devices, pair_lo=lo, pair_hi=hi)
        p = np.arange(lo, hi, dtype=np.int64)
        pi, pj = (p // C_CROSS_SLICE).astype(np.int32), (C_CROSS_SLICE + p % C_CROSS_SLICE).astype(np.int32)
        what = f"cross {devices} {name}"
        st = SR.pairs(F, pi, pj, "global")
        counts, status = SR.counts_matrix(st, torch_ops)
        assert np.array_equal(got["status"], status), what
        assert bits_equal(got["raw"], torch_ops.to_numpy(st["raw"])), f"{what}: raw"
        assert bits_equal(got["taumax"], torch_ops.to_numpy(st["taumax"])), f"{what}: taumax"
        ok = status == 0
        check_oracle(xy, pi[ok], pj[ok], got["pvalue"][ok], got["completeness"][ok], "global", what)
    _release(torch_ops)


# ---------------------------------------------------------------- 3. full walks past 2^31
@pytest.fixture(scope="module")
def d1_ref(d1, torch_ops):
    x, planted = d1
    F = SR.Features(x, torch_ops)
    r1 = _timed("reference D1 pass 1 (hist, M, top-k)", reference_walk, F, "global", topk=("abs", "signed"))
    assert r1["M"] == 1.0 and r1["hist"].sum() == P_WALK
    s_thr = threshold_from_hist(r1["hist"])
    t = s_thr / K
    r2 = _timed("reference D1 pass 2 (edges)", reference_walk, F, "global", M=1.0, t_cor=t)
    _release(torch_ops)
    return dict(hist=r1["hist"], M=1.0, t=t, s_thr=s_thr, edges=r2["edges"], abs=r1["abs"], signed=r1["signed"])


def test_d1_planted_pairs_straddle_2_31(d1, d1_ref):
    """the edges really sit where the walk's indices cross 2^31 and in the last window"""
    x, planted = d1
    i, j = d1_ref["edges"][:2]
    p = i.astype(np.int64) * (2 * C_WALK - i.astype(np.int64) - 1) // 2 + j - i - 1
    for a, b in ((2 ** 31 - 40, 2 ** 31), (2 ** 31, 2 ** 31 + 40), ((P_WALK - 1) // W * W, P_WALK)):
        assert ((p >= a) & (p < b)).sum() >= 5, f"no edge in [{a}, {b})"


@pytest.mark.parametrize("scale_max", [True, False])
def test_d1_edges_every_pair(d1, d1_ref, scale_max, torch_ops):
    x, _ = d1
    got = _timed(f"run_edges D1 scale_max={scale_max}", ik.run_edges, x, (), min_abs_cor=d1_ref["t"],
                 scale_max=scale_max)
    check_edges(got, d1_ref["edges"], 1.0, scale_max, f"D1 edges scale_max={scale_max}")
    if scale_max:
        check_oracle(x, got["i"], got["j"], got["pvalue"], got["completeness"], "global", "D1 edges")
    _release(torch_ops)


def test_d1_edges_three_devices(d1, d1_ref, torch_ops):
    x, _ = d1
    got = _timed("run_edges D1 devices=[0, 0, 0]", ik.run_edges, x, (), min_abs_cor=d1_ref["t"],
                 devices=[0, 0, 0])
    check_edges(got, d1_ref["edges"], 1.0, True, "D1 edges devices=[0, 0, 0]")
    _release(torch_ops)


@pytest.fixture(scope="module")
def p_table(torch_ops):
    """the library's p-value of a complete tie-free pair of 40 rows for every |S| (0..K): p depends on |S| alone
    there.  Column 0 is 0..39, column d + 1 a permutation with d inversions, so S = K - 2d."""
    base = np.arange(N, dtype=np.float64)
    cols = [base]
    for d in range(K + 1):
        perm, left = [], d
        rest = list(range(N))
        for pos in range(N):  # Lehmer code: take the element with min(left, remaining - 1) smaller ones after it
            c = min(left, len(rest) - 1)
            perm.append(rest.pop(c))
            left -= c
        cols.append(np.array(perm, dtype=np.float64))
    x = np.asfortranarray(np.stack(cols, axis=1))
    r = ik.run_pairs(x, (), pi=np.zeros(K + 1, dtype=np.int32), pj=np.arange(1, K + 2, dtype=np.int32),
                     want_counts=True)
    S = K - 2 * r["counts"][:, 0]
    assert np.array_equal(S, K - 2 * np.arange(K + 1))
    table = np.empty(K + 1)
    table[np.abs(S)] = r["pvalue"]
    return table


def padj_groups(hist, table):
    """(p, first rank a, last rank b) of every distinct p-value among the pairs, ascending, from the |S| histogram"""
    s = np.nonzero(hist)[0]
    p = table[s]
    ps = np.unique(p)
    cnt = np.array([hist[s[p == v]].sum() for v in ps], dtype=np.int64)
    b = np.cumsum(cnt)
    return ps, b - cnt + 1, b


def padj_reference(method, m, ps, a, b):
    """R's p.adjust per p-value group, in the order of operations of icikt_padj.cuh, in Python doubles"""
    dm = float(m)
    G = ps.size
    v = [0.0] * G
    if method == "bonferroni":
        v = [dm * float(p) for p in ps]
    elif method == "holm":
        run = -math.inf
        for g in range(G):
            run = max(run, float(m + 1 - int(a[g])) * float(ps[g]))
            v[g] = run
    else:
        run = math.inf
        for g in range(G - 1, -1, -1):
            if method == "hochberg":
                val = float(m + 1 - int(b[g])) * float(ps[g])
            else:  # BH
                val = (dm / float(int(b[g]))) * float(ps[g])
            run = min(run, val)
            v[g] = run
    return {float(p): (x if x < 1.0 else 1.0) for p, x in zip(ps, v)}


@pytest.mark.parametrize("method", ["bonferroni", "holm", "hochberg", "BH"])
def test_d1_padj_over_every_pair(d1, d1_ref, p_table, method, torch_ops):
    """BY is left out: its q = sum(1/k) over 2.15e9 terms in long double costs over a minute on the host."""
    x, _ = d1
    got = _timed(f"run_edges D1 p_adjust={method}", ik.run_edges, x, (), min_abs_cor=d1_ref["t"], p_adjust=method)
    check_edges(got, d1_ref["edges"], 1.0, True, f"D1 padj {method}")
    assert got["n_tests"] == P_WALK == 2151647200
    S = np.rint(np.abs(got["raw"]) * K).astype(np.int64)
    assert bits_equal(got["pvalue"], p_table[S]), f"{method}: p-values of the walk vs the |S| table"
    ps, a, b = padj_groups(d1_ref["hist"], p_table)
    assert b[-1] == P_WALK
    want = padj_reference(method, P_WALK, ps, a, b)
    exp = np.array([want[float(p)] for p in got["pvalue"]])
    assert bits_equal(got["padj"], exp), f"{method}: padj"
    _release(torch_ops)


@pytest.mark.parametrize("by", ["abs", "signed"])
def test_d1_topk_every_pair(d1, d1_ref, by, torch_ops):
    x, _ = d1
    got = _timed(f"run_topk D1 k=3 by={by}", ik.run_topk, x, (), k=K_TOP, by=by)
    check_topk(got, d1_ref[by], 1.0, x, "global", f"D1 top-k {by}")
    _release(torch_ops)


@pytest.mark.parametrize("persp", ["global", "local"])
def test_d2_edges_and_topk_every_pair(d2, persp, torch_ops):
    x = d2
    F = SR.Features(x, torch_ops)
    r1 = _timed(f"reference D2 {persp} pass 1 (M, top-k)", reference_walk, F, persp, topk=("abs",))
    M = r1["M"]
    # a threshold that keeps some 1e5 pairs: from one block's distribution of abs(raw / M)
    blk = SR.block(F.take(slice(0, 2048)), F, persp)
    v = (blk["raw"] / M).abs()
    v = v[(blk["status"] == 0) & ~v.isnan()].cpu().numpy()
    t = float(np.quantile(v, 1 - 1e-4))
    del blk
    r2 = _timed(f"reference D2 {persp} pass 2 (edges)", reference_walk, F, persp, M=M, t_cor=t)
    _release(torch_ops)
    n_edges = r2["edges"][0].size
    assert 10_000 <= n_edges <= 2_000_000, n_edges
    got = _timed(f"run_edges D2 {persp}", ik.run_edges, x, (), min_abs_cor=t, perspective=persp)
    check_edges(got, r2["edges"], M, True, f"D2 {persp} edges")
    sub = slice(None, None, max(1, n_edges // 200_000))
    check_oracle(x, got["i"][sub], got["j"][sub], got["pvalue"][sub], got["completeness"][sub], persp,
                 f"D2 {persp} edges")
    got = _timed(f"run_topk D2 {persp}", ik.run_topk, x, (), k=K_TOP, by="abs", perspective=persp)
    assert got["n_neighbors"][7] == 0 and got["n_neighbors"][C_WALK - 3] == 0
    check_topk(got, r1["abs"], M, x, persp, f"D2 {persp} top-k")
    _release(torch_ops)


CX, CY = 40000, 53700


def test_cross_edges_walk_past_2_31(torch_ops):
    assert CX * CY == 2 ** 31 + 516352
    rng = np.random.default_rng(4053)
    x, y = _perm_columns(rng, N, CX), _perm_columns(rng, N, CY)
    for p in list(range(2 ** 31 - 30, 2 ** 31 + 30)) + list(range(CX * CY - 30, CX * CY)):
        i, j = divmod(p, CY)
        yy = x[:, i].copy()
        for v in rng.integers(0, N - 1, int(rng.integers(1, 30))):
            a, b = yy == v, yy == v + 1
            yy[a], yy[b] = v + 1, v
        y[:, j] = yy
    Fx, Fy = SR.Features(x, torch_ops), SR.Features(y, torch_ops)
    r1 = _timed("reference cross pass 1 (hist)", reference_walk, Fx, "global", G=Fy)
    assert r1["M"] == 1.0 and r1["hist"].sum() == CX * CY
    t = threshold_from_hist(r1["hist"]) / K
    r2 = _timed("reference cross pass 2 (edges)", reference_walk, Fx, "global", G=Fy, M=1.0, t_cor=t)
    _release(torch_ops)
    got = _timed("run_cross_edges 40000 x 53700", ik.run_cross_edges, x, y, (), min_abs_cor=t)
    check_edges(got, r2["edges"], 1.0, True, "cross edges")
    p = got["i"].astype(np.int64) * CY + got["j"]
    assert ((p >= 2 ** 31 - 30) & (p < 2 ** 31 + 30)).sum() >= 30
    sub = slice(None, None, max(1, p.size // 200_000))
    xy = np.asfortranarray(np.hstack([x, y]))
    check_oracle(xy, got["i"][sub], CX + got["j"][sub], got["pvalue"][sub], got["completeness"][sub], "global",
                 "cross edges")
    _release(torch_ops)


# ---------------------------------------------------------------- 4. every pair of a moderate run
@pytest.mark.parametrize("persp", ["global", "local"])
def test_every_pair_counts_6000_columns(persp, torch_ops):
    rng = np.random.default_rng(6000)
    C = 6000
    x = np.round(rng.normal(size=(N, 1)) * 0.5 + rng.normal(size=(N, C)) * 1.5)
    x[x <= -2] = np.nan                       # left-censored
    x[rng.random(x.shape) < 0.05] = np.nan    # and random missing values
    x[:, 11] = np.nan
    x[:, 12] = 4.0
    x = np.asfortranarray(x)
    got = _timed(f"run_pairs 6000 columns {persp}", ik.run_pairs, x, (), want_counts=True, perspective=persp)
    F = SR.Features(x, torch_ops)
    iu = np.triu_indices(C, 1)
    off, R = 0, 512
    for i0 in range(0, C - 1, R):
        i1 = min(C - 1, i0 + R)
        st = SR.block(F.take(slice(i0, i1)), F, persp)
        rr, cc = iu[0][(iu[0] >= i0) & (iu[0] < i1)], iu[1][(iu[0] >= i0) & (iu[0] < i1)]
        P = rr.size
        sl = slice(off, off + P)
        r_t = torch_ops.t.as_tensor(rr - i0, device=torch_ops.device)
        c_t = torch_ops.t.as_tensor(cc, device=torch_ops.device)
        status = st["status"][r_t, c_t].cpu().numpy().astype(np.int32)
        assert np.array_equal(got["status"][sl], status), f"{persp} rows [{i0}, {i1}): status"
        ok = status == 0
        for k, name in enumerate(SR.COUNT_NAMES):
            want = st[name][r_t, c_t].cpu().numpy().astype(np.int64)
            assert np.array_equal(got["counts"][sl, k][ok], want[ok]), f"{persp} rows [{i0}, {i1}): {name}"
        for name in ("raw", "taumax"):
            assert bits_equal(got[name][sl], st[name][r_t, c_t].cpu().numpy()), f"{persp} rows [{i0}, {i1}): {name}"
        off += P
        del st
    assert off == got["status"].size
    _release(torch_ops)
