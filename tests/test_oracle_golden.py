"""Pins the CPU oracle (oracle/) against the reference's own golden values.

Sources (paths relative to /root/reference):
  tests/testthat/_snaps/kendall-tau.md     -> tests/golden/reference_snapshots.json
  tests/testthat/test-kendall-tau.R:5-59   deterministic known answers
plus scipy.stats.kendalltau (the algorithm the reference was translated from) as an
independent check of tau and of the tie-free asymptotic p-value.
"""
import json
import os

import numpy as np
import pytest
import scipy.stats as ss

from oracle import oracle as O
from oracle.r_rng import RRng


@pytest.fixture(scope="module")
def snaps(golden_dir):
    with open(os.path.join(golden_dir, "reference_snapshots.json")) as f:
        return json.load(f)


def test_snapshot_large_kendall(snaps):
    # test-kendall-tau.R:72-78 ; _snaps/kendall-tau.md:1-7
    r = RRng(1234)
    x, y = r.rnorm(50000), r.rnorm(50000)
    res = O.ici_kt(x, y, "global")
    s = snaps["large_kendall"]
    assert round(res.tau, 8) == s["tau"]
    assert round(res.pvalue, 8) == s["pvalue"]
    assert res.tau_max == s["tau_max"] and res.completeness == s["completeness"]


def _kt_matrix():
    r = RRng(1234)
    return r.rnorm(400).reshape(4, 100).T  # matrix(rnorm(400), nrow = 100, ncol = 4)


def test_snapshot_kt_fast_complete(snaps):
    # test-kendall-tau.R:153-186 ; _snaps/kendall-tau.md:49-68
    x = _kt_matrix()
    x[9, 0] = np.nan
    got = O.kt_fast(x, use="complete.obs")
    s = snaps["kt_fast_na_matrix_complete"]
    np.testing.assert_allclose(got["tau"], np.array(s["tau"]), rtol=6e-7, atol=0)
    np.testing.assert_allclose(got["pvalue"], np.array(s["pvalue"]), rtol=6e-7, atol=0)


def test_snapshot_kt_fast_pairwise(snaps):
    # _snaps/kendall-tau.md:70-90
    x = _kt_matrix()
    x[9, 0] = np.nan
    got = O.kt_fast(x, use="pairwise.complete.obs")
    s = snaps["kt_fast_na_matrix_pairwise"]
    np.testing.assert_allclose(got["tau"], np.array(s["tau"]), rtol=6e-7, atol=0)
    np.testing.assert_allclose(got["pvalue"], np.array(s["pvalue"]), rtol=6e-7, atol=0)
    # everything: any NA -> all NA (test-kendall-tau.R:167-169,178-180)
    ev = O.kt_fast(x, use="everything")
    assert np.isnan(ev["tau"][0, 0]) and np.isnan(ev["pvalue"][0, 0])


def test_kt_fast_matches_base_kendall():
    # test-kendall-tau.R:158-160: kt_fast(x)$tau == cor(x, method = "kendall")
    x = _kt_matrix()
    got = O.kt_fast(x)["tau"]
    for i in range(4):
        for j in range(4):
            assert got[i, j] == pytest.approx(ss.kendalltau(x[:, i], x[:, j]).statistic, abs=1e-14)


def test_snapshot_completeness(snaps):
    # test-kendall-tau.R:138-151 ; _snaps/kendall-tau.md:9-17
    r = RRng(1234)
    x = r.rnorm(5000).reshape(50, 100)  # byrow = TRUE
    idx = r.sample(5000, 40)
    xf = x.flatten(order="F")
    xf[idx - 1] = np.nan
    x = xf.reshape(50, 100, order="F")
    pc = O.pairwise_completeness(x, return_matrix=False)
    s = snaps["completeness_rows_4_6"]
    assert list(pc["s1"][3:6] + 1) == s["s1"] and list(pc["s2"][3:6] + 1) == s["s2"]
    assert list(pc["missingness"][3:6]) == s["missingness"]
    np.testing.assert_allclose(pc["completeness"][3:6], s["completeness"], rtol=0, atol=1e-15)
    # ici_kendalltau(...)$cor$completeness == pairwise_completeness(...)$completeness (:146-148)
    ik = O.ici_kendalltau(x, perspective="global", return_matrix=False)
    assert ik["raw"].size == pc["completeness"].size  # expect_equal(nrow(...), nrow(...)) :146
    np.testing.assert_allclose(ik["completeness"], pc["completeness"], rtol=0, atol=1e-15)


def test_basic_matches_base_r():
    # test-kendall-tau.R:5-32
    x = np.arange(1, 11, dtype=float)
    y = np.arange(1, 11, dtype=float)
    assert O.ici_kt(x, y).tau == pytest.approx(1.0, abs=1e-15)
    y[1] = 15
    assert O.ici_kt(x, y).tau == pytest.approx(ss.kendalltau(x, y).statistic, abs=1e-15)
    y = np.arange(10, 0, -1, dtype=float)
    assert O.ici_kt(x, y).tau == pytest.approx(-1.0, abs=1e-15)
    y[1] = 15
    assert O.ici_kt(x, y).tau == pytest.approx(ss.kendalltau(x, y).statistic, abs=1e-15)
    for alt in ("two.sided", "less", "greater"):
        ref = ss.kendalltau(x, y, method="asymptotic",
                            alternative=alt.replace(".", "-")).pvalue
        assert O.ici_kt(x, y, alternative=alt).pvalue == pytest.approx(ref, rel=1e-12)
    y[1] = np.nan
    assert O.ici_kt(x, y).completeness == pytest.approx(0.9, abs=1e-15)
    x[7] = np.nan
    assert O.ici_kt(x, y).completeness == pytest.approx(0.8, abs=1e-15)
    x[1] = np.nan
    assert O.ici_kt(x, y).completeness == pytest.approx(1 - 1 / 9, abs=1e-15)
    assert O.ici_kt(x, y, perspective="global").completeness == pytest.approx(0.8, abs=1e-15)


def test_reference_o_n2_matches_short():
    # test-kendall-tau.R:34-40
    rng = np.random.default_rng(7)
    x = np.sort(rng.normal(size=100))
    y = x + 1
    y[:20] = np.nan
    a = O.ici_kt(x, y, perspective="global")
    b = O.ici_kt_pairs(x, y, "global")
    # ici_kt_pairs always applies the continuity correction (src/kendallc.cpp:504)
    assert a.tau == pytest.approx(b[0], abs=1e-14)
    a2 = O.ici_kt(x, y, perspective="global", continuity=True)
    assert a2.pvalue == pytest.approx(b[1], rel=1e-8)


def test_bad_values():
    # test-kendall-tau.R:42-59
    rng = np.random.default_rng(3)
    x = np.sort(rng.normal(size=100))
    y = np.full(100, np.nan)
    r = O.ici_kt(x, y)
    assert r.status == 1 and all(np.isnan(r.as_vector()))
    with pytest.raises(ValueError, match="not the same length"):
        O.ici_kt(x, x[:99])
    r = O.ici_kt(x[1:2], x[1:2])
    assert r.status == 2 and "single value" in O.WARNINGS[r.status]
    r = O.ici_kt(x, np.ones(100))
    assert r.status == 3 and "single unique value" in O.WARNINGS[r.status]


def test_matrix_matches_pair():
    # test-kendall-tau.R:61-70, 223-239
    rng = np.random.default_rng(11)
    x = np.sort(rng.normal(size=100))
    y = x + 1
    y[:20] = np.nan
    m = np.column_stack([x, y])
    mc = O.ici_kendalltau(m, global_na=(np.nan,), perspective="global", scale_max=False)
    assert mc["raw"][1, 0] == O.ici_kt(x, y, "global").tau
    lc = O.ici_kendalltau(m, global_na=(np.nan,), perspective="global", scale_max=False,
                          return_matrix=False)
    assert lc["raw"].size == 3
    assert lc["raw"][0] == mc["raw"][1, 0] and lc["raw"][2] == mc["raw"][1, 1]


def test_include_only_counts():
    # test-kendall-tau.R:102-136 (structural: independent of the values)
    rng = np.random.default_rng(1234)
    x = rng.normal(size=(50, 100))
    assert (O.ici_kendalltau(x, include_only=0)["cor"] == 0).sum() == 9702
    assert (O.ici_kendalltau(x, include_only=[0, 2])["cor"] == 0).sum() == 9506
    inc = ([0], [1, 2])
    a = O.ici_kendalltau(x, include_only=inc)
    assert (a["cor"] == 0).sum() == 9896
    assert (O.ici_kendalltau(x, include_only=inc, diag_good=False)["cor"] == 0).sum() == 9996
    assert O.ici_kendalltau(x, include_only=inc, diag_good=False,
                            return_matrix=False)["raw"].size == 2
    with pytest.raises(ValueError, match="list of two vectors"):
        O.ici_kendalltau(x, include_only=([0], [1, 2], [3]), diag_good=False)
    with pytest.raises(ValueError, match="No comparisons to do."):
        O.ici_kendalltau(x, include_only=([101], [104]), diag_good=False)


def test_self_pair_known_pvalues(snaps):
    # data-independent known answers: any tie-free vector against itself
    for n, p in ((99, 1.076521e-48), (100, 3.480281e-49)):
        v = np.random.default_rng(n).normal(size=n)
        r = O.ici_kt(v, v)
        assert r.tau == 1.0
        assert r.pvalue == pytest.approx(p, rel=6e-7)


def test_pnorm_against_scipy():
    zs = np.concatenate([np.linspace(-37.4, 8.2, 2001), [-37.5192, -37.52, 37.6, 0.0, 1e-20]])
    for z in zs:
        lo, up = O.pnorm(z, True), O.pnorm(z, False)
        ref_lo, ref_up = ss.norm.cdf(z), ss.norm.sf(z)
        if z < -37.5193:
            assert lo == 0.0
        else:
            assert lo == pytest.approx(ref_lo, rel=5e-14 * max(1.0, z * z)), z
        if z > 37.5193:
            assert up == 0.0
        elif -8.2924 < z:
            assert up == pytest.approx(ref_up, rel=5e-14 * max(1.0, z * z)), z


def test_local_equals_global_counts_formula():
    """SURVEY 7.1: removing joint-NA rows leaves dis unchanged, ntie drops by b(b-1)/2."""
    rng = np.random.default_rng(5)
    for _ in range(50):
        n = int(rng.integers(5, 120))
        x = np.round(rng.normal(size=n) * 3)
        y = np.round(x + rng.normal(size=n) * 3)
        x[rng.random(n) < 0.3] = np.nan
        y[rng.random(n) < 0.3] = np.nan
        g, l = O.ici_kt(x, y, "global"), O.ici_kt(x, y, "local")
        if g.status or l.status:
            continue
        b = int((np.isnan(x) & np.isnan(y)).sum())
        assert l.dis == g.dis and l.ntie == g.ntie - b * (b - 1) // 2 and l.n_entry == n - b


def test_yeast_fixture_is_current(golden_dir):
    d = np.load(os.path.join(golden_dir, "yeast_missing.npz"))
    o = np.load(os.path.join(golden_dir, "yeast_oracle.npz"))
    data = d["data"].astype(np.float64)
    assert data.shape == (6887, 96)
    ex = data.copy()
    ex[O.setup_missing_matrix(data)] = np.nan
    k = 0  # Snf2.01 x Snf2.02, values recorded in SURVEY.md 8c
    r = O.ici_kt(ex[:, o["pi"][k]], ex[:, o["pj"][k]], "global")
    assert r.tau == o["global_raw"][k] and r.dis == 650208 and r.ntie == 19481
    assert r.xtie == 51756 and r.ytie == 79654
    assert r.tau == pytest.approx(ss.kendalltau(np.nan_to_num(ex[:, 0], nan=-1),
                                                np.nan_to_num(ex[:, 1], nan=-1)).statistic, abs=1e-14)
