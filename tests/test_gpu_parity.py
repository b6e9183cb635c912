"""GPU parity tests (run with -m gpu on the B200 box): the CUDA path, called through the C ABI,
against the CPU oracle on the same inputs, against the committed golden fixtures, and -- at the
BASELINE.json sizes -- through size-independent properties plus a sampled oracle check.

Bars: integer counts (dis, ntie, xtie, ytie, tot, n_entry, b) and status bit-exact;
tau / tau_max 1e-12 relative (north_star); completeness bit-exact; p-value
|p_gpu - p_ref| <= 1e-12 * max(1, z^2) * p_ref with the oracle's z (a normal tail is ill-conditioned
in z: d ln p / d ln z ~ z^2, SURVEY.md 7.3; z = 1 recovers the plain 1e-12 of north_star) and exact
zeros preserved.  The worst observed p-value error per test is written to
gpurun_out/pvalue_worst.json (copied to profiles/ per round).
"""
import json
import os
import warnings

import numpy as np
import pytest

import icikendalltau_b200 as ik
from icikendalltau_b200 import _lib, synth
from oracle import oracle as O
from oracle.r_rng import RRng

pytestmark = pytest.mark.gpu

COUNT_NAMES = ["dis", "ntie", "xtie", "ytie", "tot", "n_entry", "b"]


P_TOL = 1e-12
PVALUE_WORST = {}  # what -> worst |dp| / (max(1, z^2) p) seen (written out by conftest at session end)


def assert_pvalue(a, b, z, what=""):
    """|a - b| <= P_TOL * max(1, z^2) * |b|; NaN patterns and exact zeros must agree.  Without the
    oracle's z (golden fixtures) z^2 is bounded from the p-value itself: p >= exp(-z^2/2) / (z^2 + 1)."""
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    assert np.array_equal(np.isnan(a), np.isnan(b)), f"{what}: pvalue NaN pattern"
    m = ~np.isnan(b)
    a, b = a[m], b[m]
    assert np.array_equal(a == 0, b == 0), f"{what}: exact-zero p-values"
    nz = b != 0
    if not nz.any():
        return 0.0
    if z is not None:
        zz = np.maximum(1.0, np.asarray(z, dtype=np.float64)[m][nz] ** 2)
    else:
        zz = np.maximum(1.0, -2.0 * np.log(np.minimum(b[nz], 1.0)))
    err = np.abs(a[nz] - b[nz]) / (zz * np.abs(b[nz]))
    worst = float(err.max())
    PVALUE_WORST[what] = max(PVALUE_WORST.get(what, 0.0), worst)
    k = int(err.argmax())
    assert worst <= P_TOL, f"{what}: pvalue {a[nz][k]!r} vs {b[nz][k]!r}, z^2 = {zz[k]:.3g}, err/z^2 = {worst:.3g}"
    return worst


def assert_parity(got, ref, what=""):
    assert np.array_equal(got["status"], ref["status"]), what
    ok = ref["status"] == 0
    for k, nm in enumerate(COUNT_NAMES):
        assert np.array_equal(got["counts"][ok, k], ref["counts"][ok, k]), f"{what}: {nm}"
    for nm, tol in (("raw", 1e-12), ("taumax", 1e-12), ("completeness", 0.0)):
        a, b = got[nm], ref[nm]
        assert np.array_equal(np.isnan(a), np.isnan(b)), f"{what}: {nm} NaN pattern"
        m = ~np.isnan(b)
        np.testing.assert_allclose(a[m], b[m], rtol=tol, atol=0, err_msg=f"{what}: {nm}")
    assert_pvalue(got["pvalue"], ref["pvalue"], ref.get("z"), what)
    if ok.any():
        assert got["max_taumax"] == pytest.approx(np.nanmax(ref["taumax"]), rel=1e-12)
    else:
        assert np.isnan(got["max_taumax"])


def oracle_pairs(x, pi=None, pj=None, include_diag=False, global_na=(), **kw):
    ex = np.array(x, copy=True)
    if len(global_na):
        ex[O.setup_missing_matrix(ex, global_na)] = np.nan
    if pi is None:
        pi, pj = O.setup_comparisons(x.shape[1], None, not include_diag)
    return O.pair_loop(ex, pi, pj, ncore=os.cpu_count() or 1, want_counts=True, want_z=True, **kw)


def gen(n, C, kind, na, seed):
    rng = np.random.default_rng(seed)
    x = rng.normal(size=(n, 1)) + rng.normal(size=(n, C)) * 0.7
    if kind == "ties":
        x = np.round(x * 2)
    elif kind == "heavy":
        x = np.floor(np.exp(x))
    elif kind == "mixed":
        x[:, ::2] = np.round(x[:, ::2] * 3)
    if na > 0:
        x = np.where(x <= np.quantile(x, na), np.nan, x)
    return np.asfortranarray(x)


# ---------------------------------------------------------------- golden fixtures (config 1)
@pytest.mark.parametrize("persp", ["global", "local"])
def test_yeast_missing_matches_golden(golden_dir, persp):
    """BASELINE config 1: ici_kendalltau(yeast_missing), all 4560 pairs, vs committed oracle output."""
    d = np.load(os.path.join(golden_dir, "yeast_missing.npz"))
    o = np.load(os.path.join(golden_dir, "yeast_oracle.npz"))
    got = ik.run_pairs(d["data"].astype(np.float64), (np.nan, np.inf, 0.0), perspective=persp, want_counts=True)
    ref = {k: o[f"{persp}_{k}"] for k in ("raw", "pvalue", "taumax", "completeness", "status", "counts")}
    assert_parity(got, ref, f"yeast {persp}")
    # SURVEY.md 8c: Snf2.01 x Snf2.02
    if persp == "global":
        assert list(got["counts"][0, :4]) == [650208, 19481, 51756, 79654]
        assert got["raw"][0] == pytest.approx(0.943050719783801, rel=1e-12)


def test_yeast_ici_kendalltau_api(golden_dir):
    d = np.load(os.path.join(golden_dir, "yeast_missing.npz"))
    names = [str(s) for s in d["colnames"]]
    data = d["data"].astype(np.float64)
    got = ik.ici_kendalltau(data, colnames=names)
    ref = O.ici_kendalltau(data, ncore=os.cpu_count() or 1)
    for k in ("cor", "raw", "pvalue", "taumax", "completeness"):
        np.testing.assert_allclose(got[k], ref[k], rtol=1e-12, atol=0, err_msg=k)
    assert np.array_equal(got["keep"], ref["keep"])
    assert got["cor"].shape == (96, 96) and np.allclose(np.diag(got["taumax"]), 1.0)


# ---------------------------------------------------------------- reference snapshot values
def test_snapshot_kt_fast(golden_dir):
    """tests/testthat/test-kendall-tau.R:153-198 with the reference's snapshot numbers."""
    snaps = json.load(open(os.path.join(golden_dir, "reference_snapshots.json")))
    r = RRng(1234)
    x = r.rnorm(400).reshape(4, 100).T
    names = ["s1", "s2", "s3", "s4"]
    fast = ik.kt_fast(x, colnames=names)
    import scipy.stats as ss
    for i in range(4):
        for j in range(4):
            assert fast["tau"][i, j] == pytest.approx(ss.kendalltau(x[:, i], x[:, j]).statistic, abs=1e-14)
    x_na = x.copy()
    x_na[:, 0] = np.nan
    assert np.isnan(ik.kt_fast(x_na, use="complete.obs", colnames=names)["tau"]).all()
    x2 = x.copy()
    x2[9, 0] = np.nan
    ev = ik.kt_fast(x2[:, 0], x2[:, 1])
    assert np.isnan(ev["tau"]).all() and np.isnan(ev["pvalue"]).all()
    comp = ik.kt_fast(x2, use="complete.obs", colnames=names)
    s = snaps["kt_fast_na_matrix_complete"]
    np.testing.assert_allclose(comp["tau"], np.array(s["tau"]), rtol=6e-7)
    np.testing.assert_allclose(comp["pvalue"], np.array(s["pvalue"]), rtol=6e-7)
    pw = ik.kt_fast(x2, use="pairwise.complete.obs", colnames=names)
    s = snaps["kt_fast_na_matrix_pairwise"]
    np.testing.assert_allclose(pw["tau"], np.array(s["tau"]), rtol=6e-7)
    np.testing.assert_allclose(pw["pvalue"], np.array(s["pvalue"]), rtol=6e-7)
    pc = ik.kt_fast(x2[:, 0], x2[:, 1], use="complete.obs")
    pp = ik.kt_fast(x2[:, 0], x2[:, 1], use="pairwise.complete.obs")
    np.testing.assert_allclose(pc["tau"], pp["tau"], rtol=0, atol=0)
    assert fast["tau"][0, 1] > pc["tau"][0, 1]
    long = ik.kt_fast(x, return_matrix=False, colnames=names)
    assert long["tau"]["tau"][3] == fast["tau"][1, 2]  # df_out$tau[4, "tau"] == tau["s2", "s3"]


def test_snapshot_completeness(golden_dir):
    """test-kendall-tau.R:138-151 + _snaps/kendall-tau.md:9-17."""
    snaps = json.load(open(os.path.join(golden_dir, "reference_snapshots.json")))
    r = RRng(1234)
    x = r.rnorm(5000).reshape(50, 100)
    idx = r.sample(5000, 40)
    xf = x.flatten(order="F")
    xf[idx - 1] = np.nan
    x = xf.reshape(50, 100, order="F")
    names = [f"s{i + 1}" for i in range(100)]
    x_cor = ik.ici_kendalltau(x, perspective="global", return_matrix=False, colnames=names)
    x_comp = ik.pairwise_completeness(x, return_matrix=False, colnames=names)
    assert x_cor["cor"]["raw"].size == x_comp["completeness"].size
    np.testing.assert_allclose(x_cor["cor"]["completeness"], x_comp["completeness"], rtol=0, atol=1e-15)
    s = snaps["completeness_rows_4_6"]
    assert list(x_comp["s2"][3:6]) == ["s5", "s6", "s7"]
    assert list(x_comp["missingness"][3:6]) == s["missingness"]
    np.testing.assert_allclose(x_comp["completeness"][3:6], s["completeness"], atol=1e-15)


# ---------------------------------------------------------------- reference unit tests
def test_basic_kendall_tau_matches_base_r():
    """test-kendall-tau.R:5-32."""
    import scipy.stats as ss
    x = np.arange(1, 11, dtype=float)
    y = np.arange(1, 11, dtype=float)
    assert ik.ici_kt(x, y)[0] == pytest.approx(1.0, abs=1e-15)
    y[1] = 15
    assert ik.ici_kt(x, y)[0] == pytest.approx(ss.kendalltau(x, y).statistic, abs=1e-15)
    y = np.arange(10, 0, -1, dtype=float)
    assert ik.ici_kt(x, y)[0] == pytest.approx(-1.0, abs=1e-15)
    y[1] = 15
    assert ik.ici_kt(x, y)[0] == pytest.approx(ss.kendalltau(x, y).statistic, abs=1e-15)
    for alt in ("two.sided", "less", "greater"):
        ref = ss.kendalltau(x, y, method="asymptotic", alternative=alt.replace(".", "-")).pvalue
        assert ik.ici_kt(x, y, alternative=alt)[1] == pytest.approx(ref, rel=1e-12)
    y[1] = np.nan
    assert ik.ici_kt(x, y)[3] == pytest.approx(0.9, abs=1e-15)
    x[7] = np.nan
    assert ik.ici_kt(x, y)[3] == pytest.approx(0.8, abs=1e-15)
    x[1] = np.nan
    assert ik.ici_kt(x, y)[3] == pytest.approx(1 - 1 / 9, abs=1e-15)
    assert ik.ici_kt(x, y, perspective="global")[3] == pytest.approx(0.8, abs=1e-15)


def test_difference_and_reference_match_short():
    """test-kendall-tau.R:34-40: ici_kt(global) vs the O(n^2) ici_kt_pairs."""
    rng = np.random.default_rng(21)
    x = np.sort(rng.normal(size=100))
    y = x + 1
    y[:20] = np.nan
    a = ik.ici_kt(x, y, perspective="global", continuity=True)
    b = O.ici_kt_pairs(x, y, "global")
    assert a["tau"] == pytest.approx(b[0], abs=1e-14)
    assert a["pvalue"] == pytest.approx(b[1], rel=1e-8)


def test_bad_values():
    """test-kendall-tau.R:42-59."""
    rng = np.random.default_rng(3)
    x = np.sort(rng.normal(size=100))
    with warnings.catch_warnings():
        warnings.simplefilter("error")  # the all-NA case is silent
        r = ik.ici_kt(x, np.full(100, np.nan))
    assert list(r.keys()) == ["tau", "pvalue", "tau_max", "completeness"] and np.isnan(r.as_array()).all()
    with pytest.raises(ValueError, match="not the same length"):
        ik.ici_kt(x, x[:99])
    with pytest.warns(RuntimeWarning, match="vectors only have a single value"):
        assert np.isnan(ik.ici_kt(x[1:2], x[1:2]).as_array()).all()
    with pytest.warns(RuntimeWarning, match="have only a single unique value"):
        assert np.isnan(ik.ici_kt(x, np.ones(100)).as_array()).all()


def test_matrix_kendall_and_long_format():
    """test-kendall-tau.R:61-70 and :223-239."""
    rng = np.random.default_rng(11)
    x = np.sort(rng.normal(size=100))
    y = x + 1
    y[:20] = np.nan
    m = np.column_stack([x, y])
    mc = ik.ici_kendalltau(m, global_na=(np.nan,), perspective="global", scale_max=False, colnames=["x", "y"])
    assert ik.ici_kt(x, y, "global")[0] == mc["raw"][1, 0]
    lc = ik.ici_kendalltau(m, global_na=(np.nan,), perspective="global", scale_max=False,
                           return_matrix=False, colnames=["x", "y"])
    assert lc["cor"]["raw"].size == 3
    assert lc["cor"]["raw"][0] == mc["raw"][1, 0] and lc["cor"]["raw"][2] == mc["raw"][1, 1]


def test_include_only():
    """test-kendall-tau.R:102-136."""
    r = RRng(1234)
    x = r.rnorm(5000).reshape(100, 50).T  # matrix(rnorm(5000), nrow = 50, ncol = 100)
    names = [f"s{i + 1}" for i in range(100)]
    assert (ik.ici_kendalltau(x, include_only="s1", colnames=names)["cor"] == 0).sum() == 9702
    assert (ik.ici_kendalltau(x, include_only=["s1", "s3"], colnames=names)["cor"] == 0).sum() == 9506
    inc = {"s1": ["s1"], "s2": ["s2", "s3"]}
    a3 = ik.ici_kendalltau(x, include_only=inc, colnames=names)
    assert (a3["cor"] == 0).sum() == 9896
    a4 = ik.ici_kendalltau(x, include_only=(["s1", "s1"], ["s2", "s3"]), colnames=names)
    assert np.array_equal(a4["cor"], a3["cor"])
    assert (ik.ici_kendalltau(x, include_only=inc, diag_good=False, colnames=names)["cor"] == 0).sum() == 9996
    a6 = ik.ici_kendalltau(x, include_only=inc, diag_good=False, return_matrix=False, colnames=names)
    assert a6["cor"]["raw"].size == 2
    with pytest.raises(ValueError, match="list of two vectors"):
        ik.ici_kendalltau(x, include_only=(["s1"], ["s2", "s3"], ["s4"]), diag_good=False, colnames=names)
    with pytest.raises(ValueError, match="No comparisons to do."):
        ik.ici_kendalltau(x, include_only=(["s102"], ["s105"]), diag_good=False, colnames=names)
    # values of the included pairs equal the full run's
    full = ik.ici_kendalltau(x, colnames=names, scale_max=False)
    assert a3["raw"][0, 1] == full["raw"][0, 1] and a3["raw"][2, 0] == full["raw"][2, 0]


def test_check_timing_structure():
    """test-kendall-tau.R:256-265."""
    x = np.random.default_rng(1234).normal(size=(100, 40))
    chk = ik.ici_kendalltau(x, check_timing=True, colnames=[f"s{i}" for i in range(40)])
    assert chk["value"][0] == 5 and chk["value"][1] == 780


# ---------------------------------------------------------------- randomized parity vs oracle
CASES = [
    ("normal", 100, 6, 0.0), ("normal", 100, 6, 0.25), ("ties", 100, 6, 0.0), ("ties", 100, 6, 0.25),
    ("heavy", 333, 5, 0.3), ("mixed", 1000, 8, 0.2), ("ties", 33, 4, 0.2), ("normal", 2, 3, 0.0),
    ("ties", 3, 3, 0.0), ("normal", 31, 3, 0.5), ("ties", 32, 3, 0.1), ("normal", 2048, 4, 0.25),
    ("normal", 2049, 6, 0.25), ("ties", 4097, 4, 0.25), ("normal", 5000, 12, 0.2),
    ("heavy", 5000, 6, 0.2), ("mixed", 8193, 4, 0.25), ("mixed", 9000, 6, 0.25),
    ("normal", 16385, 4, 0.25), ("normal", 20000, 6, 0.25), ("heavy", 20000, 4, 0.25),
    ("mixed", 24577, 3, 0.2), ("mixed", 30000, 4, 0.25), ("heavy", 32768, 3, 0.3),
]


@pytest.mark.parametrize("kind,n,C,na", CASES)
def test_random_parity(kind, n, C, na):
    x = gen(n, C, kind, na, seed=n * 7 + C)
    for persp in ("global", "local"):
        got = ik.run_pairs(x, (), perspective=persp, want_counts=True)
        assert_parity(got, oracle_pairs(x, perspective=persp), f"{kind} n={n} {persp}")


def test_options_and_pair_lists():
    x = gen(500, 7, "mixed", 0.3, 5)
    for alt, cont in (("less", True), ("greater", False), ("two.sided", True), ("bogus", False)):
        got = ik.run_pairs(x, (), alternative=alt, continuity=cont, want_counts=True)
        assert_parity(got, oracle_pairs(x, alternative=alt, continuity=cont), alt)
    got = ik.run_pairs(x, (), include_diag=True, perspective="local", want_counts=True)
    assert_parity(got, oracle_pairs(x, include_diag=True, perspective="local"), "diag")
    pi, pj = [0, 0, 3, 6, 2, 2, 5], [1, 5, 3, 0, 4, 2, 1]
    got = ik.run_pairs(x, (), pi=pi, pj=pj, want_counts=True)
    assert_parity(got, oracle_pairs(x, np.array(pi, np.int32), np.array(pj, np.int32)), "pair list")
    got = ik.run_pairs(x, (), want_counts=True, pair_lo=5, pair_hi=17)
    full = oracle_pairs(x)
    assert_parity(got, {k: v[5:17] for k, v in full.items()}, "pair range")


def test_global_na_and_degenerate_columns():
    x = gen(500, 8, "mixed", 0.3, 9)
    x[::5, 1] = 0.0
    x[::9, 2] = np.inf
    x[::11, 2] = -np.inf
    x[:, 4] = np.nan
    x[:, 5] = 3.0
    x[:, 6] = np.where(np.arange(500) % 2 == 0, np.nan, 7.0)  # one value + missing
    for g in ((np.nan, np.inf, 0.0), (np.nan,), (), (np.nan, np.inf, 0.0, 3.0)):
        for persp in ("global", "local"):
            got = ik.run_pairs(x, g, perspective=persp, want_counts=True)
            assert_parity(got, oracle_pairs(x, global_na=g, perspective=persp), f"global_na={g} {persp}")


def test_absorbed_minimum_and_signed_zero():
    # |min| so large that min - 0.1 == min: missing rows tie with the minimum (SURVEY.md 8a row 3)
    rng = np.random.default_rng(4)
    x = rng.normal(size=(200, 4))
    x[:, 0] = np.round(x[:, 0]) * 1e17
    x[:, 1] = np.where(rng.random(200) < 0.3, -np.inf, x[:, 1])
    x[:, 2] = np.where(rng.random(200) < 0.5, -0.0, 0.0) + np.round(x[:, 2])
    x[rng.random(x.shape) < 0.2] = np.nan
    for persp in ("global", "local"):
        got = ik.run_pairs(x, (), perspective=persp, want_counts=True)
        assert_parity(got, oracle_pairs(x, perspective=persp), f"absorbed {persp}")


def test_naive_kernel_matches_tiled_and_oracle():
    x = gen(700, 9, "mixed", 0.3, 77)
    for persp in ("global", "local"):
        got = ik.run_pairs(x, (), perspective=persp, want_counts=True, kernel=_lib.KERNEL_NAIVE)
        assert_parity(got, oracle_pairs(x, perspective=persp), f"naive {persp}")


def test_pnorm_device_matches_oracle():
    z = np.concatenate([np.linspace(-38.5, 38.5, 4001), [-37.5193, 37.5193, 0.0, 1e-20, -8.2924, 8.2924,
                                                          np.inf, -np.inf, np.nan]])
    for lower in (True, False):
        dev = ik.pnorm_device(z, lower)
        ref = np.array([O.pnorm(v, lower) for v in z])
        assert np.array_equal(np.isnan(dev), np.isnan(ref))
        m = ~np.isnan(ref)
        assert np.array_equal(dev[m] == 0, ref[m] == 0)
        np.testing.assert_allclose(dev[m], ref[m], rtol=2e-13, atol=0)


def test_plan_api_device_resident_reuse():
    x = gen(3000, 10, "mixed", 0.25, 8)
    plan = ik.Plan(3000, 10, perspective="local", want_counts=True)
    plan.upload(x)
    for _ in range(3):  # repeated runs on the resident matrix give identical results
        plan.columns(())
        plan.pairs()
        got = plan.download(want_counts=True)
        assert_parity(got, oracle_pairs(x, perspective="local"), "plan")
    assert np.array_equal(plan.column_n_na(), np.isnan(x).sum(axis=0))
    t = plan.timings()
    assert t["pairs_ms"] > 0 and t["n_launches"] >= 4
    plan.close()


# ---------------------------------------------------------------- BASELINE.json sizes
def _sampled_oracle_check(x, persp, got, n_sample=48, seed=0, what="sampled"):
    C = x.shape[1]
    pi, pj = O.setup_comparisons(C, None, True)
    sel = np.random.default_rng(seed).choice(pi.size, size=min(n_sample, pi.size), replace=False)
    ref = O.pair_loop(x, pi[sel], pj[sel], perspective=persp, ncore=os.cpu_count() or 1, want_counts=True,
                      want_z=True)
    sub = {k: (v[sel] if isinstance(v, np.ndarray) else v) for k, v in got.items()}
    sub["max_taumax"] = np.nanmax(ref["taumax"])  # the global max is checked separately
    assert_parity(sub, ref, what)
    return pi, pj, sel


def test_config2_full_size():
    """BASELINE config 2: 5000 features x 100 samples, 20% left-censored, global; all 4950 pairs."""
    x, persp = synth.make("config2")
    got = ik.run_pairs(x, (), perspective=persp, want_counts=True)
    assert_parity(got, oracle_pairs(x, perspective=persp), "config2")


def _shape_invariants(x, persp, got, pi, pj, n_swap=64, gna=()):
    """Size-independent properties at full size: |tau| <= tau_max, every pair computed, and the counts
    of a spread of pairs are unchanged when the two columns swap roles (the kernel treats them
    asymmetrically: one is staged, the other streamed)."""
    assert (got["status"] == 0).all()
    assert (np.abs(got["raw"]) <= got["taumax"] * (1 + 1e-15)).all()
    assert got["max_taumax"] == np.nanmax(got["taumax"])
    sel = np.linspace(0, pi.size - 1, n_swap).astype(np.int64)
    sw = ik.run_pairs(x, gna, pi=pj[sel], pj=pi[sel], perspective=persp, want_counts=True)
    for k in (0, 1, 4, 5, 6):  # dis, ntie, tot, n_entry, b (xtie/ytie swap with the columns)
        assert np.array_equal(sw["counts"][:, k], got["counts"][sel, k]), COUNT_NAMES[k]
    assert np.array_equal(sw["counts"][:, 2], got["counts"][sel, 3])
    assert np.array_equal(sw["raw"], got["raw"][sel])


def test_config3_full_size():
    """BASELINE config 3 at FULL size: 20000 features x 1000 samples, 25% left-censored, local +
    scale_max; all 499,500 pairs on the GPU, 1000 sampled pairs against the oracle."""
    x, persp = synth.make("config3")
    assert x.shape == (20000, 1000) and persp == "local"
    got = ik.run_pairs(x, (), perspective=persp, want_counts=True)
    assert got["raw"].size == 499500
    pi, pj, _ = _sampled_oracle_check(x, persp, got, n_sample=1000, what="config3 full")
    _shape_invariants(x, persp, got, pi, pj)
    # tiled kernel == naive kernel (independent Fenwick algorithm) on a slice of the pair order
    nv = ik.run_pairs(x, (), perspective=persp, want_counts=True, kernel=_lib.KERNEL_NAIVE,
                      pair_lo=100000, pair_hi=100400)
    assert np.array_equal(nv["counts"], got["counts"][100000:100400])
    # scale_max: cor = raw / max(taumax) through the R-level API (matrix path on the device)
    names = [f"s{i}" for i in range(x.shape[1])]
    res = ik.ici_kendalltau(x, global_na=(np.nan,), perspective="local", colnames=names)
    assert res["cor"][0, 1] == got["raw"][0] / got["max_taumax"]
    assert res["raw"][999, 998] == got["raw"][-1]


def test_config5_full_size():
    """BASELINE config 5 at FULL size: 2000 features x 5000 samples, 12,497,500 pairs, global;
    1200 sampled pairs against the oracle."""
    x, persp = synth.make("config5")
    assert x.shape == (2000, 5000)
    got = ik.run_pairs(x, (), perspective=persp, want_counts=True)
    assert got["raw"].size == 12497500
    pi, pj, _ = _sampled_oracle_check(x, persp, got, n_sample=1200, what="config5 full")
    _shape_invariants(x, persp, got, pi, pj)
    # identical columns: tau == 1, dis == 0
    x2 = np.asfortranarray(np.column_stack([x[:, 0], x[:, 0], x[:, 1]]))
    r = ik.run_pairs(x2, (), want_counts=True)
    assert r["raw"][0] == 1.0 and r["counts"][0, 0] == 0


def test_target_full_size():
    """north_star target at FULL size: 20000 features x 2000 samples, 25% censored, global;
    1,999,000 pairs, 1000 sampled pairs against the oracle (counts bit-exact, tau 1e-12)."""
    x, persp = synth.make("target")
    assert x.shape == (20000, 2000)
    got = ik.run_pairs(x, (), perspective=persp, want_counts=True)
    assert got["raw"].size == 1999000
    pi, pj, _ = _sampled_oracle_check(x, persp, got, n_sample=1000, what="target full")
    _shape_invariants(x, persp, got, pi, pj)
    # several devices inside one call (sharded K1 + peer gather of the tables when there are peers)
    ndev = _lib.load().icikt_device_count()
    if ndev > 1:
        many = ik.run_pairs(x, (), perspective=persp, want_counts=True, devices=list(range(ndev)))
        for k in ("raw", "pvalue", "taumax", "completeness", "status", "counts"):
            np.testing.assert_array_equal(got[k], many[k], err_msg=k)


def test_config4_full_size():
    """BASELINE config 4 at FULL size: adenocarcinoma-shaped counts, 60000 features x 200 samples,
    zeros missing, heavy ties, global; 19,900 pairs, 1000 sampled pairs against the oracle."""
    x, persp = synth.make("config4")
    assert x.shape == (60000, 200)
    gna = (np.nan, np.inf, 0.0)
    got = ik.run_pairs(x, gna, perspective=persp, want_counts=True)
    assert got["raw"].size == 19900
    pi, pj, _ = _sampled_oracle_check(x, persp, got, n_sample=1000, what="config4 full")
    _shape_invariants(x, persp, got, pi, pj, gna=gna)


def test_int32_overflow_domain_is_reported():
    """SURVEY.md 8a: the reference's integer intermediates are int32 (Rcpp IntegerVector); a tie group
    of >= 1024 rows overflows count_rank_tie's t1 sum and one of >= 1292 rows its t0 sum (signed-overflow UB,
    not a specification).  The GPU path follows the exact int64 oracle; this test runs the oracle's
    emulate_int32 mode beside it on a 1500-wide missing group and RECORDS what the wrap does to the
    reference's own p-value (gpurun_out/int32_domain.json) instead of hiding it."""
    rng = np.random.default_rng(99)
    n = 6000
    x = np.asfortranarray(rng.normal(size=(n, 2)) + rng.normal(size=(n, 1)) * 0.05)
    x[np.argsort(x[:, 0])[:1500], 0] = np.nan
    x[np.argsort(x[:, 1])[:1100], 1] = np.nan
    x[rng.permutation(n)[:3000], 1] = rng.normal(size=3000)  # weaken the correlation: a p-value away from 0
    got = ik.run_pairs(x, (), perspective="global", want_counts=True)
    exact = O.pair_loop(x, [0], [1], perspective="global", want_counts=True, want_z=True)
    wrap = O.pair_loop(x, [0], [1], perspective="global", want_counts=True, want_z=True, emulate_int32=True)
    assert_parity(got, exact, "int32 domain, exact oracle")
    # counts and tau stay inside the int32 domain here, the variance terms do not
    assert np.array_equal(exact["counts"], wrap["counts"])
    assert exact["raw"][0] == wrap["raw"][0]
    report = {"n": n, "na_group_x": int(np.isnan(x[:, 0]).sum()), "na_group_y": int(np.isnan(x[:, 1]).sum()), "tau": float(exact["raw"][0]),
              "z_exact": float(exact["z"][0]), "z_emulate_int32": float(wrap["z"][0]),
              "pvalue_gpu": float(got["pvalue"][0]), "pvalue_exact_oracle": float(exact["pvalue"][0]),
              "pvalue_emulate_int32": float(wrap["pvalue"][0]),
              "note": "GPU == exact oracle; the emulate_int32 column is what the reference's own int32 "
                      "arithmetic yields for the same vectors"}
    os.makedirs(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpurun_out"), exist_ok=True)
    with open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpurun_out",
                           "int32_domain.json"), "w") as f:
        json.dump(report, f, indent=1)
    assert wrap["z"][0] != exact["z"][0], "the 1500-wide group must leave the int32 domain of the variance sums"


def test_sharded_columns_plan_api_matches_full_run():
    """Sharded K1 through the plan API: two plans (two ranks' worth, here on one device) each
    preprocess half of the columns, exchange the table slices icikt_plan_tables describes with
    plain device copies, and then produce their halves of the pair order; together they must equal
    the single-plan run bit for bit.  Under torchrun the same exchange goes through NCCL
    (sharding.exchange_tables, exercised by bench.py --gpus N)."""
    import torch
    from icikendalltau_b200 import sharding
    x = gen(9000, 21, "mixed", 0.25, seed=4242)  # 9000 rows: the multi-kernel column path
    xs = gen(3000, 21, "heavy", 0.3, seed=4243)  # 3000 rows: the fused column kernel
    for mat in (x, xs):
        n, C = mat.shape
        P = C * (C - 1) // 2
        ref = ik.run_pairs(mat, (), perspective="local", want_counts=True)
        plans = []
        for r in range(2):
            lo, hi = sharding.pair_range(P, r, 2)
            pl = ik.Plan(n, C, perspective="local", want_counts=True, pair_lo=lo, pair_hi=hi)
            c0, c1 = sharding.column_range(C, r, 2)
            pl.upload_columns(np.asfortranarray(mat), c0, c1)
            pl.columns_range((), c0, c1)
            pl.sync()
            plans.append(pl)
        dev = torch.device("cuda", 0)
        for r in range(2):  # pull the other rank's slices
            o = 1 - r
            c0, c1 = sharding.column_range(C, o, 2)
            for (pm, bpc), (po, _) in zip(plans[r].tables(), plans[o].tables()):
                dst = torch.as_tensor(sharding._DevBytes(pm, bpc * C), device=dev)
                src = torch.as_tensor(sharding._DevBytes(po, bpc * C), device=dev)
                dst[c0 * bpc:c1 * bpc].copy_(src[c0 * bpc:c1 * bpc])
        torch.cuda.synchronize()
        parts = []
        for pl in plans:
            pl.columns_finish()
            pl.pairs()
            parts.append(pl.download(want_counts=True))
        for k in ("raw", "pvalue", "taumax", "completeness", "status", "counts"):
            np.testing.assert_array_equal(np.concatenate([q[k] for q in parts]), ref[k], err_msg=k)
        assert sharding.combine_max_taumax([q["max_taumax"] for q in parts]) == ref["max_taumax"]
        for pl in plans:
            pl.close()


# ---------------------------------------------------------------- long vectors (global-scratch variant)
def test_snapshot_large_kendall(golden_dir):
    """test-kendall-tau.R:72-78 + _snaps/kendall-tau.md:1-7: n = 50000, set.seed(1234)."""
    snaps = json.load(open(os.path.join(golden_dir, "reference_snapshots.json")))["large_kendall"]
    r = RRng(1234)
    x, y = r.rnorm(50000), r.rnorm(50000)
    v = ik.ici_kt(x, y, perspective="global")
    assert round(v["tau"], 8) == snaps["tau"] and round(v["pvalue"], 8) == snaps["pvalue"]
    assert v["tau_max"] == 1.0 and v["completeness"] == 1.0


def test_big_kendall_matches_o_n2_reference():
    """test-kendall-tau.R:80-89 (the reference's long test): n = 50000 with 5000 missing."""
    rng = np.random.default_rng(50)
    x = np.sort(rng.normal(size=50000))
    y = x + 1
    x[:5000] = np.nan
    t1 = ik.ici_kt(x, y, perspective="global", continuity=True)
    t2 = O.ici_kt_pairs(x, y, "global")
    assert t1["tau"] == pytest.approx(t2[0], abs=1e-14)
    assert t1["pvalue"] == pytest.approx(t2[1], rel=1e-8)


@pytest.mark.parametrize("kind,n,C,na", [("normal", 40000, 3, 0.25), ("mixed", 50000, 4, 0.25),
                                         ("heavy", 60000, 3, 0.4), ("normal", 65535, 3, 0.1),
                                         ("ties", 65535, 2, 0.3)])
def test_long_vectors(kind, n, C, na):
    x = gen(n, C, kind, na, seed=n + C)
    for persp in ("global", "local"):
        got = ik.run_pairs(x, (), perspective=persp, want_counts=True)
        assert_parity(got, oracle_pairs(x, perspective=persp), f"{kind} n={n} {persp}")


def test_too_long_is_refused():
    x = np.random.default_rng(0).normal(size=(65536, 2))
    with pytest.raises(ik.IciktError) as e:
        ik.run_pairs(x)
    assert e.value.code == _lib.ERR_TOO_LONG


@pytest.mark.parametrize("kind,n,C,na", [("mixed", 1000, 6, 0.25), ("heavy", 5000, 4, 0.3),
                                         ("normal", 20000, 3, 0.25)])
def test_forced_global_scratch_matches(kind, n, C, na, monkeypatch):
    """The global-scratch code path on sizes where the shared-memory path is the default."""
    x = gen(n, C, kind, na, seed=3 * n + C)
    ref = oracle_pairs(x, perspective="local")
    monkeypatch.setenv("ICIKT_FORCE_GMEM", "1")
    got = ik.run_pairs(x, (), perspective="local", want_counts=True)
    assert_parity(got, ref, f"forced gmem {kind} n={n}")


@pytest.mark.gpu
@pytest.mark.parametrize("n,fracs,ties", [(3000, (0.85, 0.0, 0.4, 0.97), False), (256, (255 / 256, 0.0, 0.5), False),
                                          (5000, (0.7, 0.1, 0.0), True), (20000, (0.9, 0.02, 0.3), True)])
def test_uneven_missingness_first_group_emission(n, fracs, ties):
    """Columns with very different missing fractions: the rank histogram of x's first group does not
    fit beside its output slots and is processed in several rounds (or in the spare words); with ties
    in y long runs go through the cooperative list.  Both orders of every pair are exercised."""
    rng = np.random.default_rng(n)
    base = rng.normal(size=n)
    cols = []
    for fr in fracs:
        v = base + 0.5 * rng.normal(size=n)
        if ties:
            v = np.round(v * 1.5)
        k = int(round(fr * n))
        if k:
            v[np.argsort(v)[:k]] = np.nan
        cols.append(v)
    x = np.asfortranarray(np.column_stack(cols))
    C = x.shape[1]
    pi = np.array([i for i in range(C) for j in range(C) if i != j], dtype=np.int32)
    pj = np.array([j for i in range(C) for j in range(C) if i != j], dtype=np.int32)
    for persp in ("global", "local"):
        got = ik.run_pairs(x, (), pi=pi, pj=pj, perspective=persp, want_counts=True)
        assert_parity(got, oracle_pairs(x, pi=pi, pj=pj, perspective=persp), f"uneven NA n={n} {persp}")


def _oracle_complete(x, pi, pj):
    """kt_split with use = 'pairwise.complete.obs' (R/kendalltau.R:323-341): drop the rows missing in
    either column, then ici_kt on what is left."""
    P = len(pi)
    out = dict(raw=np.full(P, np.nan), pvalue=np.full(P, np.nan), taumax=np.full(P, np.nan), z=np.full(P, np.nan),
               status=np.zeros(P, dtype=np.int32), counts=np.zeros((P, 7), dtype=np.int64))
    for k in range(P):
        good = ~np.isnan(x[:, pi[k]]) & ~np.isnan(x[:, pj[k]])
        if good.sum() == 0:
            out["status"][k] = 1
            continue
        sub = np.asfortranarray(np.column_stack([x[good, pi[k]], x[good, pj[k]]]))
        r = O.pair_loop(sub, np.array([0], np.int32), np.array([1], np.int32), perspective="local",
                        want_counts=True, want_z=True)
        out["status"][k] = r["status"][0]
        for nm in ("raw", "pvalue", "taumax", "z"):
            out[nm][k] = r[nm][0]
        out["counts"][k] = r["counts"][0]
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("kind,n,C,na", [("normal", 300, 7, 0.2), ("ties", 1000, 6, 0.3), ("heavy", 2500, 5, 0.35),
                                         ("mixed", 6000, 5, 0.25), ("normal", 33, 5, 0.5), ("ties", 20000, 3, 0.4)])
def test_complete_observations_mode(kind, n, C, na):
    """Device-side pairwise.complete.obs: every count on the shared rows is bit-exact against the
    oracle run on the filtered vectors; includes (i,i) pairs, both orders and degenerate columns."""
    x = gen(n, C, kind, na, seed=7 * n + C)
    rng = np.random.default_rng(n)
    x[rng.random(n) < 0.1, 1] = np.nan          # missingness that is not left-censoring
    x = np.column_stack([x, np.full(n, np.nan), np.full(n, 2.5), np.where(np.arange(n) % 3 == 0, np.nan, 1.0)])
    x[0, 2] = np.nan                             # a column with exactly one missing row
    x = np.asfortranarray(x)
    C = x.shape[1]
    pi = np.array([i for i in range(C) for j in range(C)], dtype=np.int32)
    pj = np.array([j for i in range(C) for j in range(C)], dtype=np.int32)
    got = ik.run_pairs(x, (), pi=pi, pj=pj, perspective="complete", want_counts=True)
    ref = _oracle_complete(x, pi, pj)
    assert np.array_equal(got["status"], ref["status"])
    ok = ref["status"] == 0
    for k, nm in enumerate(COUNT_NAMES[:6]):
        assert np.array_equal(got["counts"][ok, k], ref["counts"][ok, k]), nm
    for nm, tol in (("raw", 1e-12), ("taumax", 1e-12)):
        a, b = got[nm], ref[nm]
        assert np.array_equal(np.isnan(a), np.isnan(b)), nm
        m = ~np.isnan(b)
        np.testing.assert_allclose(a[m], b[m], rtol=tol, atol=0, err_msg=nm)
    assert_pvalue(got["pvalue"], ref["pvalue"], ref["z"], f"complete {kind} n={n}")
    assert np.all(got["completeness"][ok] == 1.0)


@pytest.mark.gpu
def test_kt_fast_pairwise_uses_device_mode_and_matches_host_filtering():
    x = gen(800, 9, "mixed", 0.3, seed=99)
    names = [f"s{i}" for i in range(x.shape[1])]
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        fast = ik.kt_fast(x, use="pairwise.complete.obs", colnames=names)
    ref = O.kt_fast(x, use="pairwise.complete.obs")
    np.testing.assert_allclose(fast["tau"], ref["tau"], rtol=1e-12, equal_nan=True)
    assert_pvalue(fast["pvalue"], ref["pvalue"], None, "kt_fast pairwise")


@pytest.mark.gpu
def test_chunked_copy_out_of_large_result_sets(monkeypatch):
    """Result sets above the one-shot staging limit leave the device through two pinned chunks;
    forced here with tiny limits so that every array takes several chunks of uneven length."""
    x = gen(400, 40, "mixed", 0.25, seed=5)
    ref = oracle_pairs(x, perspective="global")
    monkeypatch.setenv("ICIKT_STAGE_ALL", "1024")
    monkeypatch.setenv("ICIKT_STAGE_CHUNK", "1000")
    _lib.release_workspace()
    got = ik.run_pairs(x, (), perspective="global", want_counts=True)
    _lib.release_workspace()
    assert_parity(got, ref, "chunked copy-out")


@pytest.mark.gpu
def test_multi_gpu_call_matches_single_gpu():
    """icikt_all_pairs_multi: the pair order sliced over the devices inside one call gives the very
    bytes of the single-device call (with one GPU the two slices simply run on the same device)."""
    ndev = _lib.load().icikt_device_count()
    x = gen(700, 23, "mixed", 0.25, seed=77)
    one = ik.run_pairs(x, (), perspective="local", include_diag=True, want_counts=True)
    devices = [0, 1 % ndev, 0] if ndev > 1 else [0, 0, 0]
    many = ik.run_pairs(x, (), perspective="local", include_diag=True, want_counts=True, devices=devices)
    for k in ("raw", "pvalue", "taumax", "completeness", "status", "counts"):
        np.testing.assert_array_equal(one[k], many[k], err_msg=k)
    assert one["max_taumax"] == many["max_taumax"]
    res = ik.ici_kendalltau(x, global_na=(np.nan,), colnames=[f"s{i}" for i in range(23)], n_gpus=min(2, max(ndev, 1)))
    ref = ik.ici_kendalltau(x, global_na=(np.nan,), colnames=[f"s{i}" for i in range(23)])
    np.testing.assert_array_equal(res["cor"], ref["cor"])


@pytest.mark.gpu
def test_random_small_matrices_all_modes():
    """Many small random matrices with every mix of ties, missingness, constant / all-missing columns:
    all three modes against the oracle.  Group sizes straddle the large-tie threshold (128) so that
    direct comparison, in-place histogram sort and the first-group emission all take part."""
    rng = np.random.default_rng(int(os.environ.get("ICIKT_TEST_SEED", "20240611")))
    for case in range(60):
        n = int(rng.choice([2, 3, 5, 17, 64, 129, 130, 257, 400, 900]))
        C = int(rng.integers(2, 7))
        levels = int(rng.choice([1, 2, 3, 6, 20, 1000]))
        x = rng.normal(size=(n, C))
        x = np.round(x * levels / 3.0) if levels < 1000 else x
        for c in range(C):
            frac = float(rng.choice([0.0, 0.0, 0.1, 0.5, 0.9, 1.0]))
            x[rng.random(n) < frac, c] = np.nan
        x = np.asfortranarray(x)
        pi = np.array([i for i in range(C) for j in range(C)], dtype=np.int32)
        pj = np.array([j for i in range(C) for j in range(C)], dtype=np.int32)
        for persp in ("global", "local"):
            got = ik.run_pairs(x, (), pi=pi, pj=pj, perspective=persp, want_counts=True)
            assert_parity(got, oracle_pairs(x, pi=pi, pj=pj, perspective=persp), f"case {case} n={n} {persp}")
        got = ik.run_pairs(x, (), pi=pi, pj=pj, perspective="complete", want_counts=True)
        ref = _oracle_complete(x, pi, pj)
        assert np.array_equal(got["status"], ref["status"]), f"case {case} complete status"
        ok = ref["status"] == 0
        for k, nm in enumerate(COUNT_NAMES[:6]):
            assert np.array_equal(got["counts"][ok, k], ref["counts"][ok, k]), f"case {case} complete {nm}"
        np.testing.assert_allclose(got["raw"][ok], ref["raw"][ok], rtol=1e-12, atol=0)
        assert_pvalue(got["pvalue"][ok], ref["pvalue"][ok], ref["z"][ok], "small matrices complete")


@pytest.mark.gpu
def test_repeated_runs_are_identical():
    """The pair kernel uses shared-memory atomics, a dynamic work queue and block-wide barriers: the
    integer counts of repeated runs must be bit-identical (a race would show up as a flaky count)."""
    x = gen(3000, 40, "mixed", 0.25, seed=11)
    x[:, 5] = np.round(x[:, 5])            # a column with large tie groups next to continuous ones
    first = ik.run_pairs(x, (), perspective="local", want_counts=True)
    for _ in range(15):
        again = ik.run_pairs(x, (), perspective="local", want_counts=True)
        for k in ("counts", "status", "raw", "pvalue", "taumax", "completeness"):
            np.testing.assert_array_equal(first[k], again[k], err_msg=k)


# ---------------------------------------------------------------- result formats on the device
def host_matrices(x, global_na, scale_max, diag_good, pi=None, pj=None, **kw):
    """scale_and_reshape (R/kendalltau.R:357-421) done on the host from the per-pair arrays."""
    n, C = x.shape
    if pi is None:
        r = ik.run_pairs(x, global_na, include_diag=not diag_good, **kw)
        pi, pj = O.setup_comparisons(C, None, diag_good)
    else:
        r = ik.run_pairs(x, global_na, pi=pi, pj=pj, **kw)
    raw = r["raw"]
    cols = dict(cor=raw / r["max_taumax"] if scale_max else raw.copy(), raw=raw, pvalue=r["pvalue"],
                taumax=r["taumax"], completeness=r["completeness"])
    out = {}
    excl = O.setup_missing_matrix(x, global_na) if len(global_na) else np.zeros(x.shape, dtype=bool)
    n_good = (~excl).sum(axis=0)
    for k, v in cols.items():
        m = np.zeros((C, C))
        m[pi, pj] = v
        m[pj, pi] = v
        if diag_good:
            dg = {"cor": n_good / n_good.max(), "raw": n_good / n_good.max(), "pvalue": np.zeros(C),
                  "taumax": np.ones(C), "completeness": n_good / n}[k]
            m[np.arange(C), np.arange(C)] = dg
        out[k] = m
    return out, r, n_good


@pytest.mark.gpu
@pytest.mark.parametrize("scale_max,diag_good", [(True, True), (True, False), (False, True), (False, False)])
def test_device_matrix_fill_matches_host_reshape(scale_max, diag_good):
    x = gen(700, 23, "mixed", 0.2, seed=31)
    x[:, 5] = 3.0  # a constant column: degenerate pairs, NaN entries, a warning class
    gna = (np.nan, np.inf, 0.0)
    ref, r, n_good = host_matrices(x, gna, scale_max, diag_good, perspective="global")
    got = _lib.run_matrices(x, gna, scale_max, diag_good, n_good, perspective="global")
    for k in _lib.MATRIX_NAMES:
        assert np.array_equal(got[k], ref[k], equal_nan=True), k
        assert np.array_equal(got[k], got[k].T, equal_nan=True), k
    hist = np.bincount(r["status"], minlength=_lib.NSTATUS)
    assert list(got["status_counts"]) == list(hist)
    # degenerate pairs carry R's NA_real_ bit pattern (low word 1954), so an R binder needs no fix-up
    assert got["raw"].view(np.uint64)[5, 0] == 0x7FF00000000007A2 and got["cor"].view(np.uint64)[0, 5] == 0x7FF00000000007A2
    assert got["max_taumax"] == r["max_taumax"]
    # n_good from the device's own missing counts (global_na holds NaN, so they agree)
    got2 = _lib.run_matrices(x, gna, scale_max, diag_good, None, perspective="global", want=("cor", "completeness"))
    assert set(got2) & set(_lib.MATRIX_NAMES) == {"cor", "completeness"}
    for k in ("cor", "completeness"):
        assert np.array_equal(got2[k], ref[k], equal_nan=True), k


@pytest.mark.gpu
def test_device_matrix_fill_pair_list_and_chunked_copy(monkeypatch):
    x = gen(500, 40, "ties", 0.25, seed=32)
    rng = np.random.default_rng(7)
    pi_all, pj_all = O.setup_comparisons(40, None, True)
    sel = np.sort(rng.choice(pi_all.size, size=300, replace=False))
    pi, pj = pi_all[sel].astype(np.int32), pj_all[sel].astype(np.int32)
    ref, r, n_good = host_matrices(x, (), True, True, pi=pi, pj=pj, perspective="local")
    got = _lib.run_matrices(x, (), True, True, n_good, pi=pi, pj=pj, perspective="local")
    for k in _lib.MATRIX_NAMES:
        assert np.array_equal(got[k], ref[k], equal_nan=True), k
    assert (got["raw"] == 0).sum() >= 40 * 40 - 2 * 300 - 40  # pairs that were not asked for stay 0
    # matrices above the staging limit leave the device through the two pinned chunks
    monkeypatch.setenv("ICIKT_STAGE_ALL", "1024")
    monkeypatch.setenv("ICIKT_STAGE_CHUNK", "1000")
    _lib.release_workspace()
    ref, r, n_good = host_matrices(x, (), True, False, perspective="global")
    got = _lib.run_matrices(x, (), True, False, n_good, perspective="global")
    _lib.release_workspace()
    for k in _lib.MATRIX_NAMES:
        assert np.array_equal(got[k], ref[k], equal_nan=True), k


@pytest.mark.gpu
def test_ici_kendalltau_matrix_path_matches_long_format():
    x = gen(900, 17, "heavy", 0.3, seed=33)
    names = [f"s{i}" for i in range(17)]
    for diag_good in (True, False):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            m = ik.ici_kendalltau(x, colnames=names, diag_good=diag_good)
            l = ik.ici_kendalltau(x, colnames=names, diag_good=diag_good, return_matrix=False)["cor"]
        idx = {s: k for k, s in enumerate(names)}
        i = np.array([idx[s] for s in l["s1"]]); j = np.array([idx[s] for s in l["s2"]])
        for k in ("cor", "raw", "pvalue", "taumax", "completeness"):
            assert np.array_equal(m[k][i, j], l[k], equal_nan=True), k
            assert np.array_equal(m[k][j, i], l[k], equal_nan=True), k


@pytest.mark.gpu
@pytest.mark.parametrize("gna", [(np.nan, np.inf, 0.0), (0.0,), (np.inf, 2.0, 3.0), ()])
def test_pairwise_completeness_kernel(gna):
    x = gen(1000, 19, "heavy", 0.2, seed=34)
    x[5, 3] = np.inf
    x[7, 4] = -np.inf
    excl = O.setup_missing_matrix(x, gna) if len(gna) else np.zeros(x.shape, dtype=bool)
    pi, pj = O.setup_comparisons(19, None, False)
    miss = np.array([(excl[:, a] | excl[:, b]).sum() for a, b in zip(pi, pj)])
    r = _lib.pairwise_completeness(x, gna, want_matrix=True)
    assert np.array_equal(r["missing"], miss)
    assert np.array_equal(r["completeness"], 1 - miss / 1000)
    m = np.zeros((19, 19))
    m[pi, pj] = 1 - miss / 1000
    m[pj, pi] = 1 - miss / 1000
    assert np.array_equal(r["matrix"], m)
    sel = np.array([3, 50, 7, 7, 120])
    r2 = _lib.pairwise_completeness(x, gna, pi=pj[sel], pj=pi[sel])  # either order
    assert np.array_equal(r2["missing"], miss[sel])
    names = [f"s{i}" for i in range(19)]
    assert np.array_equal(ik.pairwise_completeness(x, gna, colnames=names), m)
    long = ik.pairwise_completeness(x, gna, colnames=names, include_only="s3", return_matrix=False)
    keep = (pi == 3) | (pj == 3)
    assert np.array_equal(long["missingness"], miss[keep])


@pytest.mark.gpu
@pytest.mark.parametrize("scale_max,diag_good", [(True, True), (False, False), (True, False)])
def test_multi_gpu_matrices_match_single_gpu(scale_max, diag_good):
    """icikt_matrices_multi: the pair order sliced over the devices, every device filling and returning
    its own block of columns (reading the other devices' per-pair results in place), gives the very
    bytes of the single-device matrices -- incl. NA_real_ for degenerate pairs, the diag_good diagonal
    and the status counts.  With one GPU the slices run on the same device."""
    ndev = _lib.load().icikt_device_count()
    x = gen(900, 37, "mixed", 0.25, seed=123)
    x[:, 11] = 3.0      # a constant column: status 3 in a whole row/column of every matrix
    x[:, 30] = np.nan   # an all-missing one: status 1
    gna = (np.nan, np.inf, 0.0)
    n_good = (~O.setup_missing_matrix(x, gna)).sum(axis=0)
    one = _lib.run_matrices(x, gna, scale_max, diag_good, n_good, perspective="local")
    for devices in ([0, 1 % ndev, 0], list(range(ndev)) if ndev > 1 else [0, 0], [0, 0, 0, 0, 0]):
        many = _lib.run_matrices(x, gna, scale_max, diag_good, n_good, perspective="local", devices=devices)
        for k in _lib.MATRIX_NAMES:
            assert np.array_equal(one[k].view(np.uint64), many[k].view(np.uint64)), (k, devices)
        assert np.array_equal(one["status_counts"], many["status_counts"]), devices
        assert one["max_taumax"] == many["max_taumax"]
    # n_good derived by the library (n - missing rows) when the caller passes none
    a = _lib.run_matrices(x, (), scale_max, diag_good, None, perspective="global")
    b = _lib.run_matrices(x, (), scale_max, diag_good, None, perspective="global", devices=[0, 0, 0])
    for k in _lib.MATRIX_NAMES:
        assert np.array_equal(a[k].view(np.uint64), b[k].view(np.uint64)), k
    # and through the R-level API
    names = [f"s{i}" for i in range(x.shape[1])]
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        r1 = ik.ici_kendalltau(x, colnames=names)
        r2 = ik.ici_kendalltau(x, colnames=names, n_gpus=max(2, min(ndev, 8)) if ndev > 1 else 1)
    for k in _lib.MATRIX_NAMES:
        assert np.array_equal(r1[k], r2[k], equal_nan=True), k


@pytest.mark.gpu
@pytest.mark.parametrize("n", [3000, 12000, 30000])
def test_sort_high_word_collisions(n):
    """K1 sorts the keys' high 32 bits and repairs neighbours with equal high words against the low words;
    long runs fall back to the full 64-bit sort.  Columns built to hit every branch, in all three sort
    variants (fused n <= 8192, shared-memory n <= 22528, global): values that differ ONLY in the low word
    (one run as long as the column -> fallback), clusters of 2..11 such values inside ordinary data (repair),
    integers (low word zero: ties, nothing to repair), plus missing values."""
    rng = np.random.default_rng(n)
    eps = 2.0 ** -45
    c0 = 1.0 + eps * rng.permutation(n)                         # all high words equal, all values distinct
    c1 = rng.normal(size=n)
    for start in range(0, n - 16, 97):                          # clusters that share a high word
        k = int(rng.integers(2, 12))
        c1[start:start + k] = c1[start] * (1.0 + eps * rng.permutation(k))
    c2 = np.floor(np.exp(rng.normal(size=n) * 2.0))             # counts
    c3 = rng.normal(size=n)
    c4 = np.where(rng.random(n) < 0.5, 3.0 + eps * rng.integers(0, 6, size=n), rng.normal(size=n))  # short runs + ties
    x = np.column_stack([c0, c1, c2, c3, c4])
    x[rng.random(x.shape) < 0.15] = np.nan
    x = np.asfortranarray(x)
    for persp in ("global", "local"):
        got = ik.run_pairs(x, (), perspective=persp, want_counts=True)
        assert_parity(got, oracle_pairs(x, perspective=persp), f"high-word collisions n={n} {persp}")


@pytest.mark.gpu
def test_staged_pageable_upload_matches_plain_copy(monkeypatch):
    """Matrices of 8 MB and more in pageable host memory are uploaded through the plan's two pinned chunks by
    several host threads (staged_copy_in); the results must be the bytes of the plain cudaMemcpy2DAsync path,
    also when the matrix is larger than one chunk and the last chunk is ragged."""
    x = gen(1300, 900, "mixed", 0.2, seed=31337)  # 9.4 MB
    monkeypatch.setenv("ICIKT_STAGE_CHUNK", str(3 << 20))  # several chunks, ragged tail
    _lib.release_workspace()
    a = ik.run_pairs(x, (), perspective="local", pair_lo=0, pair_hi=5000)
    monkeypatch.setenv("ICIKT_NO_STAGED_UPLOAD", "1")
    _lib.release_workspace()
    b = ik.run_pairs(x, (), perspective="local", pair_lo=0, pair_hi=5000)
    _lib.release_workspace()
    for k in ("raw", "pvalue", "taumax", "completeness", "status"):
        np.testing.assert_array_equal(a[k], b[k], err_msg=k)
    assert a["max_taumax"] == b["max_taumax"]


def _same_pairs(a, b, what):
    for k in ("raw", "pvalue", "taumax", "completeness", "status", "counts"):
        if k in a or k in b:
            np.testing.assert_array_equal(a[k], b[k], err_msg=f"{what}: {k}")
    assert a["max_taumax"] == b["max_taumax"] or (np.isnan(a["max_taumax"]) and np.isnan(b["max_taumax"])), what


@pytest.mark.gpu
@pytest.mark.parametrize("persp,diag,kind", [("global", False, "mixed"), ("local", True, "ties"),
                                             ("complete", False, "mixed")])
def test_pipelined_one_shot_matches_plain_call(monkeypatch, persp, diag, kind):
    """Large all-pairs jobs go through the pipelined call (column chunks uploaded while earlier chunks are
    computed, row blocks copied out while later ones run; icikt_stage_table).  Forced on for a small matrix it
    must return the bytes of the plain upload -> columns -> pairs -> download sequence, through both result
    paths (one pinned mirror / two pinned chunks) and for pageable and pinned input."""
    import torch
    x = gen(900, 300, kind, 0.2, seed=4242)
    kw = dict(perspective=persp, include_diag=diag, want_counts=True)
    monkeypatch.setenv("ICIKT_NO_PIPELINE", "1")
    _lib.release_workspace()
    plain = ik.run_pairs(x, (), **kw)
    if persp != "complete":  # (the complete-observations mode is checked against kt_fast's own tests)
        assert_parity(plain, oracle_pairs(x, perspective=persp, include_diag=diag), f"plain {persp}")
    monkeypatch.delenv("ICIKT_NO_PIPELINE")
    monkeypatch.setenv("ICIKT_PIPELINE_MIN_BYTES", "1")
    _lib.release_workspace()
    piped = ik.run_pairs(x, (), **kw)
    _same_pairs(piped, plain, f"pipelined {persp}")
    assert piped["timings"]["n_launches"] > plain["timings"]["n_launches"], "the pipelined path did not run"
    one = ik.run_pairs(x, (), devices=[0], **kw)  # icikt_all_pairs_multi with one device: the same pipelined call
    _same_pairs(one, plain, f"pipelined, devices=[0] {persp}")
    assert one["timings"]["n_launches"] == piped["timings"]["n_launches"], "devices=[0] did not take the pipelined path"
    again = ik.run_pairs(x, (), **kw)  # the cached staged plan, second use
    _same_pairs(again, plain, f"pipelined, cached plan {persp}")
    xp = torch.from_numpy(np.asfortranarray(x).T.copy()).pin_memory().numpy().T  # pinned, column-major
    _same_pairs(ik.run_pairs(xp, (), **kw), plain, f"pipelined, pinned input {persp}")
    monkeypatch.setenv("ICIKT_STAGE_ALL", "1000")       # results through the two pinned chunks ...
    monkeypatch.setenv("ICIKT_STAGE_CHUNK", str(40000))  # ... several chunks per block and array
    monkeypatch.setenv("ICIKT_PIPELINE_BLOCKS", "3")
    _lib.release_workspace()
    _same_pairs(ik.run_pairs(x, (), **kw), plain, f"pipelined, chunked results {persp}")
    _lib.release_workspace()


@pytest.mark.gpu
def test_pipelined_matrices_match_plain_call(monkeypatch):
    x = gen(800, 260, "mixed", 0.25, seed=777)
    monkeypatch.setenv("ICIKT_NO_PIPELINE", "1")
    _lib.release_workspace()
    plain = _lib.run_matrices(x, (), perspective="global", diag_good=False)
    monkeypatch.delenv("ICIKT_NO_PIPELINE")
    monkeypatch.setenv("ICIKT_PIPELINE_MIN_BYTES", "1")
    _lib.release_workspace()
    piped = _lib.run_matrices(x, (), perspective="global", diag_good=False)
    _lib.release_workspace()
    for k in _lib.MATRIX_NAMES:
        np.testing.assert_array_equal(piped[k], plain[k], err_msg=k)
    np.testing.assert_array_equal(piped["status_counts"], plain["status_counts"])
    assert piped["max_taumax"] == plain["max_taumax"]


@pytest.mark.gpu
@pytest.mark.parametrize("n", [700, 9000, 30000])
def test_first_group_bitmap_fallback_on_shared_ranks(n):
    """The first-group emission keeps one BIT per rank of the other column when that column is nearly tie-free
    (fewer than n/8 tied rows); two rows of the group that do share a rank must send the pair through the
    counter path instead.  Columns: x left-censored, y continuous except for a few duplicated values planted on
    rows that are missing in x (the collision), z with its duplicates on rows present in x (no collision), w with
    its minimum tied and no missing rows (rank 0 is a real value there)."""
    rng = np.random.default_rng(n)
    base = rng.normal(size=n)
    x = base + 0.3 * rng.normal(size=n)
    x[x < np.quantile(x, 0.3)] = np.nan
    miss = np.flatnonzero(np.isnan(x))
    pres = np.flatnonzero(~np.isnan(x))
    y = base + 0.5 * rng.normal(size=n)
    y[miss[1:40:2]] = y[miss[0:39:2][: len(miss[1:40:2])]]       # pairs of equal values inside x's missing rows
    y[miss[50:53]] = y[miss[49]]                                  # and one run of four
    y[rng.choice(n, n // 10, replace=False)] = np.nan             # y has missing rows of its own (rank 0 = missing)
    z = base + 0.5 * rng.normal(size=n)
    z[pres[1:40:2]] = z[pres[0:39:2][: len(pres[1:40:2])]]
    w = rng.normal(size=n)
    w[miss[:5]] = w.min() - 1.0                                   # five rows of x's first group share w's lowest rank
    data = np.asfortranarray(np.stack([x, y, z, w, base], axis=1))
    for persp in ("global", "local"):
        got = ik.run_pairs(data, (), perspective=persp, want_counts=True)
        assert_parity(got, oracle_pairs(data, perspective=persp), f"bitmap fallback n={n} {persp}")
