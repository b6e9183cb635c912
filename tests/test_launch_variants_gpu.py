"""Every launch variant of the pair kernel (K2), reached on purpose and checked bit for bit against the CPU
oracle: the launch tier (0, 1, 2) that K1's device-side maxima select, pass B of tier 2 and the large-group sort
beside it in the same launch, every warp count W a launch shape accepts (with the zero compaction of tier 0 on
and off), the benchmark's own many-units shapes on small matrices, the three register classes, the shared-memory
and global-scratch forms, and tier escalation inside the pipelined call and across sharded K1.

The variant is pinned with the library's own knobs (ICIKT_WARPS, ICIKT_REGCLASS, ICIKT_FORCE_GMEM,
ICIKT_PIPELINE_MIN_BYTES); `_lib.launch_shape` reads the same environment and shows what was honoured.  Which
tier and which per-pair path a dataset takes is computed from K1's statistics read back from the device, after
those statistics are checked against a NumPy restatement: a later change of a threshold cannot quietly stop
these tests from reaching pass B."""
import numpy as np
import pytest

import icikendalltau_b200 as ik
from icikendalltau_b200 import _lib, sharding, synth
from tests.test_gpu_parity import _oracle_complete, _same_pairs, assert_parity, oracle_pairs

pytestmark = pytest.mark.gpu

# icikt_common.cuh: kLargeTie, kDirectBudget; icikt_pairs.cu: the pass-B budget (16 n) of the tier choice
LARGE_TIE, DIRECT_BUDGET, PASS_B_BUDGET = 128, 24, 16
KNOBS = ("ICIKT_WARPS", "ICIKT_REGCLASS", "ICIKT_FORCE_GMEM", "ICIKT_PIPELINE_MIN_BYTES", "ICIKT_NO_PIPELINE",
         "ICIKT_LARGE_TIE", "ICIKT_DIRECT_BUDGET")

# ColStats (icikt_common.cuh), 64 bytes per column
STATS = np.dtype([("n_na", "<i4"), ("first_run", "<i4"), ("n_tied", "<i4"), ("n_groups", "<i4"), ("levels", "<i4"),
                  ("g0extra", "<i4"), ("flags", "<i4"), ("n_tgroups", "<i4"), ("s2o", "<i8"), ("s3o", "<i8"),
                  ("s5o", "<i8"), ("cconst", "<u8")])
STATS_TABLE = 8  # its index in icikt_plan_tables


@pytest.fixture
def knobs(monkeypatch):
    """knobs(NAME=value, ...) sets (None: removes) tuning knobs; the cached plans are dropped before and after
    every change, so the next call plans its launches with them."""
    for k in KNOBS:
        monkeypatch.delenv(k, raising=False)
    _lib.release_workspace()

    def set_knobs(**kv):
        for k, v in kv.items():
            if v is None:
                monkeypatch.delenv(k, raising=False)
            else:
                monkeypatch.setenv(k, str(v))
        _lib.release_workspace()

    yield set_knobs
    _lib.release_workspace()


# ---------------------------------------------------------------- K1's statistics, restated
def host_stats(v):
    """ColStats of one column as K1 defines them (everything but cconst): groups in ascending order, the NA group
    first (it takes the minimum's rows too when min - 0.1 == min); large groups are groups g >= 1 of >= 128 rows,
    counted only when the sum of their squared sizes exceeds 24 n."""
    n = v.size
    miss = np.isnan(v)
    a = int(miss.sum())
    vals, sizes = np.unique(v[~miss], return_counts=True)
    sizes = [int(s) for s in sizes]
    absorb = 0 < a < n and vals[0] - 0.1 == vals[0]
    if a == 0:
        groups = sizes
    elif absorb:
        groups = [a + sizes[0]] + sizes[1:]
    else:
        groups = [a] + sizes
    g = np.array(groups, dtype=np.int64)
    K = g.size
    rest = g[1:]
    big = rest[rest >= LARGE_TIE]
    n_large = big.size if int((big * big).sum()) > DIRECT_BUDGET * n else 0
    o = g[1:] if a > 0 else g
    return dict(n_na=a, first_run=int(g[0]) if g[0] > 1 else 0, n_tied=int(rest[rest > 1].sum()), n_groups=K,
                levels=max(1, (K - 1).bit_length()), g0extra=int(g[0]) - a if a > 0 else 0,
                flags=int(absorb) | (n_large << 8), n_tgroups=int((rest > 1).sum()),
                s2o=int((o * (o - 1)).sum()), s3o=int((o * (o - 1) * (o - 2)).sum()),
                s5o=int((o * (o - 1) * (2 * o + 5)).sum()))


def device_stats(x):
    """K1's ColStats table of x, copied from the device after Plan.upload + Plan.columns"""
    import torch
    n, C = x.shape
    pl = ik.Plan(n, C)
    try:
        pl.upload(x)
        pl.columns()
        pl.sync()
        ptr, bpc = pl.tables()[STATS_TABLE]
        assert bpc == STATS.itemsize
        raw = torch.as_tensor(sharding._DevBytes(ptr, bpc * C), device=torch.device("cuda", 0)).cpu().numpy()
    finally:
        pl.close()
    return raw.view(STATS)


def checked_stats(x):
    """the device's statistics of every column, after checking each field but cconst against host_stats"""
    dev = device_stats(x)
    for c in range(x.shape[1]):
        want = host_stats(x[:, c])
        got = {k: int(dev[k][c]) for k in want}
        assert got == want, f"column {c}: device {got} != host {want}"
    return dev


def tier_of(st, n):
    """the launch tier the pair kernel's device-side maxima select"""
    nlg = int((st["flags"] >> 8).max())
    if nlg == 0:
        return 0
    return 2 if nlg * int(st["n_groups"].max()) > PASS_B_BUDGET * n else 1


def n_large(st):
    return (st["flags"] >> 8).astype(np.int64)


def by_pass_b(st, n, tier, pi, pj):
    """per pair: pass B takes x's tied rows (x = pj, the column the kernel does not stage)"""
    nlg = n_large(st)[pj]
    return (nlg > 0) & (tier == 2) & (nlg * st["n_groups"][pi].astype(np.int64) > PASS_B_BUDGET * n)


def compacts(st, n, W, kk, pi, pj):
    """per pair: whether the tier-0 kernel with zero compaction (shared memory, W >= 8) leaves y's rank-0 keys out
    of pass A (icikt_pairs.cu, `cz = ...`)"""
    kkc = 8 * kk
    fr = st["first_run"].astype(np.int64)
    y0 = np.maximum(fr[pi], 1)
    lead = np.minimum(fr[pj], y0)
    return ((n - y0 + kkc - 1) // kkc + 31) // 32 < W - lead // kkc // 32


def all_pairs(C):
    pi, pj = np.triu_indices(C, 1)
    return pi.astype(np.int32), pj.astype(np.int32)


def ordered_pairs(C):
    pi, pj = np.nonzero(~np.eye(C, dtype=bool))
    return pi.astype(np.int32), pj.astype(np.int32)


def check(x, pi=None, pj=None, persps=("global", "local"), naive=False, what=""):
    """the tiled kernel against the oracle (and the one-thread-per-pair kernel), counts and status bit for bit;
    returns the runs by perspective"""
    out = {}
    for persp in persps:
        got = ik.run_pairs(x, (), pi=pi, pj=pj, perspective=persp, want_counts=True)
        assert_parity(got, oracle_pairs(x, pi=pi, pj=pj, perspective=persp), f"{what} {persp}")
        if naive:
            nv = ik.run_pairs(x, (), pi=pi, pj=pj, perspective=persp, want_counts=True, kernel=_lib.KERNEL_NAIVE)
            np.testing.assert_array_equal(got["status"], nv["status"], err_msg=f"{what} {persp}: naive status")
            np.testing.assert_array_equal(got["counts"], nv["counts"], err_msg=f"{what} {persp}: naive counts")
        out[persp] = got
    return out


# ---------------------------------------------------------------- data
def distinct_col(rng, n, K):
    """n rows holding exactly K distinct values 0 .. K-1 (the other n - K rows repeat some: small tie groups)"""
    v = np.concatenate([np.arange(K), rng.integers(0, K, n - K)]).astype(np.float64)
    return rng.permutation(v)


def grouped_col(rng, n, n_big, size, n_na=0, absorbed=False):
    """n_na missing rows, n_big tie groups of `size` rows above the rest, which holds nearly distinct values
    (a tenth of them repeated: small tie groups as well)"""
    rest = n - n_na - n_big * size
    low = distinct_col(rng, rest, max(1, rest - rest // 10))
    v = np.concatenate([np.full(n_na, np.nan), low, np.repeat(rest + 10.0 + np.arange(n_big), size)])
    if absorbed:
        v = 1e17 + 1024.0 * v  # min - 0.1 == min: the missing rows tie with the minimum
    return rng.permutation(v)


def with_missing(rng, v, n_na):
    v = v.copy()
    v[rng.permutation(v.size)[:n_na]] = np.nan
    return v


def tier2_matrix(n, n_big, size, seed):
    """Columns (n_big * K_y against 16 n decides pass B per pair; x is the later column of a pair):
    H   n_big groups of `size` rows, K_H small;      D1  K = floor(16 n / n_big): the large-group sort for x = H;
    D2  K = D1 + 1: pass B for x = H;                 S   a rounded normal, a few large groups, never pass B;
    HL  H left-censored (a large first group);        D2M D2 with missing rows of its own (the NA group in K);
    HA  HL absorbed (min - 0.1 == min);               DA  absorbed with K = D1 + 1;
    N   a continuous column with missing rows.
    HL and HA hold as many of the large groups as fit beside their missing rows."""
    rng = np.random.default_rng(seed)
    kb = PASS_B_BUDGET * n // n_big
    na = n // 20
    n_big_l = min(n_big, (n - 2 * na - 100) // size)
    cols = dict(H=grouped_col(rng, n, n_big, size),
                D1=distinct_col(rng, n, kb),
                D2=distinct_col(rng, n, kb + 1),
                S=np.round(rng.standard_normal(n)),
                HL=grouped_col(rng, n, n_big_l, size, n_na=2 * na),
                D2M=np.concatenate([np.full(na, np.nan), distinct_col(rng, n - na, kb)]),
                HA=grouped_col(rng, n, n_big_l, size, n_na=na, absorbed=True),
                DA=np.concatenate([np.full(na, np.nan), 1e17 + 1024.0 * distinct_col(rng, n - na, kb + 1)]),
                N=with_missing(rng, rng.standard_normal(n), n // 4))
    cols["D2M"] = rng.permutation(cols["D2M"])
    cols["DA"] = rng.permutation(cols["DA"])
    return list(cols), np.asfortranarray(np.column_stack(list(cols.values())))


def censored(n, missing, seed, extra=()):
    """left-censored columns of one shared signal: column c has its missing[c] lowest rows missing"""
    rng = np.random.default_rng(seed)
    base = rng.standard_normal(n)
    cols = []
    for a in missing:
        v = base + 0.5 * rng.standard_normal(n)
        if a:
            v[np.argsort(v)[:a]] = np.nan
        cols.append(v)
    return np.asfortranarray(np.column_stack(cols + list(extra)))


# ---------------------------------------------------------------- 1. statistics and tiers
def test_k1_statistics_and_tiers(knobs):
    """K1's statistics against their restatement, and the tier they select, on one dataset of each kind the
    other tests rely on: tier 0, tier 1 (shared memory and in place), tier 2 (shared memory and global scratch)"""
    rng = np.random.default_rng(1)
    cases = []
    x = censored(3000, [0, 5, 900, 2999, 1500], seed=2)
    cases.append(("tier 0", x, 0, "smem"))
    x = np.asfortranarray(np.column_stack([grouped_col(rng, 6000, 10, 300), with_missing(rng, np.round(rng.standard_normal(6000) * 3), 700),
                                           rng.standard_normal(6000)]))
    cases.append(("tier 1", x, 1, "smem"))
    x = np.asfortranarray(np.column_stack([grouped_col(rng, 60000, 10, 400, n_na=5000), rng.standard_normal(60000)]))
    cases.append(("tier 1 long", x, 1, "inplace"))
    cases.append(("tier 2", tier2_matrix(4096, 17, 200, seed=3)[1], 2, "smem"))
    cases.append(("tier 2 long", tier2_matrix(30000, 60, 200, seed=4)[1], 2, "gmem"))
    absorbed = 1e17 + 1024.0 * rng.integers(0, 3000, size=(4000, 3)).astype(np.float64)
    absorbed[rng.random(absorbed.shape) < 0.25] = np.nan
    absorbed[:, 2] = np.nan  # all missing
    cases.append(("absorbed / all missing", np.asfortranarray(absorbed), 0, "smem"))
    for what, x, tier, variant in cases:
        st = checked_stats(x)
        n = x.shape[0]
        assert tier_of(st, n) == tier, what
        assert _lib.launch_shape(n, tier)["variant"] == variant, what


# ---------------------------------------------------------------- 2. tier 2 and pass B
@pytest.mark.parametrize("n,n_big,size", [(4096, 17, 200), (20000, 40, 200), (30000, 60, 200), (65535, 511, 128)])
def test_tier2_pass_b(knobs, n, n_big, size):
    """Tier 2 in shared memory (n = 4 096, 20 000) and on the global scratch (30 000, 65 535; at 65 535 a column
    with 511 large groups, the most the 512-slot group table is asked to hold).  Every ordered pair of one launch:
    pass B, the large-group sort exactly at the per-pair boundary (n_big * K_y = 16 n or just below), pairs without
    large groups; x with a large first group, y with missing rows of its own, absorbed columns."""
    names, x = tier2_matrix(n, n_big, size, seed=n)
    st = checked_stats(x)
    assert tier_of(st, n) == 2
    col = {nm: k for k, nm in enumerate(names)}
    assert n_large(st)[col["H"]] == n_big
    W = _lib.launch_shape(n, 2)["warps"]  # the shape of a large job (a few pairs would plan their own)
    knobs(ICIKT_WARPS=W)
    assert _lib.launch_shape(n, 2)["variant"] == ("smem" if n <= 20000 else "gmem")
    pi, pj = ordered_pairs(len(names))
    pb = by_pass_b(st, n, 2, pi, pj)
    sort = (n_large(st)[pj] > 0) & ~pb
    h = col["H"]
    assert pb[(pj == h) & (pi == col["D2"])].all() and sort[(pj == h) & (pi == col["D1"])].all()
    assert pb[(pj == h) & (pi == col["D2M"])].all() and pb[(pj == h) & (pi == col["DA"])].all()  # y: NA group in K
    for x_name in ("HL", "HA"):  # x with a large first group (left-censored / absorbed)
        assert pb[pj == col[x_name]].any() and sort[pj == col[x_name]].any()
    assert (n_large(st)[pj] == 0).any()
    check(x, pi, pj, naive=n <= 4096, what=f"tier 2 n={n} W={W}")


def test_tier2_complete_observations(knobs):
    """the complete-observations mode on the tier-2 matrix: pass B on the rows both columns have"""
    n = 4096
    names, x = tier2_matrix(n, 17, 200, seed=11)
    keep = [k for k, nm in enumerate(names) if nm not in ("HA", "DA")]  # absorbed columns: host path (status 9)
    names, x = [names[k] for k in keep], np.asfortranarray(x[:, keep])
    st = checked_stats(x)
    assert tier_of(st, n) == 2
    pi, pj = ordered_pairs(len(names))
    assert by_pass_b(st, n, 2, pi, pj).any()
    got = ik.run_pairs(x, (), pi=pi, pj=pj, perspective="complete", want_counts=True)
    ref = _oracle_complete(x, pi, pj)
    np.testing.assert_array_equal(got["status"], ref["status"])
    ok = ref["status"] == 0
    np.testing.assert_array_equal(got["counts"][ok, :6], ref["counts"][ok, :6])
    np.testing.assert_allclose(got["raw"][ok], ref["raw"][ok], rtol=1e-12, atol=0)


def test_small_groups_before_a_four_bit_pass_a(knobs):
    """Long vectors (y's ranks read from global memory): x's small tie groups are compared on the gathered
    sequence itself, and with y of at most 16 distinct values pass A is its low-nibble level alone, which
    parks each warp's totals over the first keys of its range.  The comparison has to be finished everywhere
    first; the same pair, repeated, must give the oracle's counts every time."""
    n = 65535
    rng = np.random.default_rng(31)
    x = np.asfortranarray(np.column_stack([np.round(rng.standard_normal(n)), distinct_col(rng, n, 2051)]))
    st = checked_stats(x)
    assert st["n_groups"][0] <= 16 and st["n_tied"][1] > n // 2 and n_large(st)[1] == 0
    assert _lib.launch_shape(n, tier_of(st, n))["variant"] == "gmem"
    pi, pj = np.zeros(64, np.int32), np.ones(64, np.int32)
    ref = oracle_pairs(x, pi=pi[:1], pj=pj[:1])
    got = ik.run_pairs(x, (), pi=pi, pj=pj, want_counts=True)
    np.testing.assert_array_equal(got["status"], np.repeat(ref["status"], 64))
    np.testing.assert_array_equal(got["counts"], np.repeat(ref["counts"], 64, axis=0))


# ---------------------------------------------------------------- 3. tier escalation across the matrix
def test_pipelined_call_escalates_to_tier2(knobs):
    """Pipelined one-shot call on 130 columns with the tie-heavy column last: the launches before its chunk see
    tier-0 maxima, the last one tier 2.  Bytes equal the plain call's, counts the oracle's."""
    n, C = 4096, 130
    rng = np.random.default_rng(12)
    x = np.asfortranarray(np.column_stack([with_missing(rng, rng.standard_normal((n, C - 1)).ravel(), n)
                                           .reshape(n, C - 1), grouped_col(rng, n, 17, 200)]))
    st = checked_stats(x)
    assert tier_of(st[:C - 1], n) == 0 and tier_of(st, n) == 2
    _, launches = _lib.stage_table(C)  # the plan's stage table (148 SMs, 8 row blocks)
    assert launches[-1, 1] == C and (launches[:, 1] < C).any()
    knobs(ICIKT_NO_PIPELINE=1)
    plain = ik.run_pairs(x, (), want_counts=True)
    knobs(ICIKT_NO_PIPELINE=None, ICIKT_PIPELINE_MIN_BYTES=1)
    piped = ik.run_pairs(x, (), want_counts=True)
    assert piped["timings"]["n_launches"] > plain["timings"]["n_launches"], "the pipelined path did not run"
    _same_pairs(piped, plain, "pipelined vs plain")
    pi, pj = all_pairs(C)
    sel = np.flatnonzero((pj >= C - 2) | (np.arange(pi.size) % 37 == 0))
    ref = oracle_pairs(x, pi=pi[sel], pj=pj[sel])
    np.testing.assert_array_equal(piped["status"][sel], ref["status"])
    ok = ref["status"] == 0
    np.testing.assert_array_equal(piped["counts"][sel][ok], ref["counts"][ok])


def test_sharded_k1_escalates_to_tier2(knobs):
    """Sharded K1 (two plans, table exchange as in test_gpu_parity): one half holds the large groups (tier 1
    alone), the other the many distinct values (tier 0 alone); only the maxima over all columns after the exchange
    select tier 2.  The two halves of the pair order together equal the single-plan run bit for bit."""
    import torch
    n = 4096
    names, x = tier2_matrix(n, 17, 200, seed=13)
    order = ["H", "S", "HL", "HA", "D1", "D2", "D2M", "N"]
    x = np.asfortranarray(x[:, [names.index(nm) for nm in order]])
    C = x.shape[1]
    st = checked_stats(x)
    halves = [sharding.column_range(C, r, 2) for r in range(2)]
    assert [tier_of(st[lo:hi], n) for lo, hi in halves] == [1, 0] and tier_of(st, n) == 2
    P = C * (C - 1) // 2
    for persp in ("global", "local"):
        ref = ik.run_pairs(x, (), perspective=persp, want_counts=True)
        assert_parity(ref, oracle_pairs(x, perspective=persp), f"sharded reference {persp}")
        plans = []
        for r in range(2):
            lo, hi = sharding.pair_range(P, r, 2)
            pl = ik.Plan(n, C, perspective=persp, want_counts=True, pair_lo=lo, pair_hi=hi)
            pl.upload_columns(x, *halves[r])
            pl.columns_range((), *halves[r])
            pl.sync()
            plans.append(pl)
        dev = torch.device("cuda", 0)
        for r in range(2):
            c0, c1 = halves[1 - r]
            for (pm, bpc), (po, _) in zip(plans[r].tables(), plans[1 - r].tables()):
                dst = torch.as_tensor(sharding._DevBytes(pm, bpc * C), device=dev)
                src = torch.as_tensor(sharding._DevBytes(po, bpc * C), device=dev)
                dst[c0 * bpc:c1 * bpc].copy_(src[c0 * bpc:c1 * bpc])
        torch.cuda.synchronize()
        parts = []
        for pl in plans:
            pl.columns_finish()
            pl.pairs()
            parts.append(pl.download(want_counts=True))
            pl.close()
        for k in ("raw", "pvalue", "taumax", "completeness", "status", "counts"):
            np.testing.assert_array_equal(np.concatenate([q[k] for q in parts]), ref[k], err_msg=f"{persp} {k}")


# ---------------------------------------------------------------- 4. every warp count
def sweep_lengths(n, R):
    """y-present counts len' (rows of y outside its lowest group): k R - 1, k R, k R + 1, and the first two and
    last two multiples of 32 R (a warp's range)"""
    lens = {n - 1}
    for k in (1, 2, n // R - 1):
        for d in (-1, 0, 1):
            lens.add(k * R + d)
    m = list(range(32 * R, n, 32 * R))
    lens.update(m[:2] + m[-2:])
    return sorted((v for v in lens if 2 <= v <= n - 1), reverse=True)


@pytest.mark.parametrize("n,tier", [(3000, 0), (20000, 0), (20000, 2)])
def test_every_warp_count(knobs, n, tier):
    """Every W (1 .. 32) launch_shape accepts at n, forced with ICIKT_WARPS, on left-censored columns whose
    y-present counts fall around multiples of that shape's thread range R = 8 kk and at multiples of 32 R.  Tier 0:
    at every W >= 8, some pairs run pass A on the compacted sequence and some do not, wherever the shape leaves room
    for both.  Tier 2 adds a column of 40 large groups, last, so that it is x in pass B for every other column."""
    ran, cache = [], {}
    for W in range(1, 33):
        knobs(ICIKT_WARPS=W)
        shape = _lib.launch_shape(n, tier)
        if shape["warps"] != W:
            assert W < 3, f"n={n}: W={W} refused"
            continue
        kk = shape["runs"]
        ran.append(W)
        if kk not in cache:
            lens = sweep_lengths(n, 8 * kk)
            extra = [grouped_col(np.random.default_rng(kk), n, 40, 200)] if tier == 2 else []
            x = censored(n, [n - v if v < n - 1 else 0 for v in lens], seed=kk, extra=extra)
            st = checked_stats(x)
            assert tier_of(st, n) == tier
            C = x.shape[1]
            pi, pj = all_pairs(C)
            fr = st["first_run"]
            assert sorted(n - np.maximum(fr[:len(lens)], 1)) == sorted(lens)
            ref = {p: oracle_pairs(x, perspective=p) for p in ("global", "local")}
            cache[kk] = (x, st, pi, pj, ref)
        x, st, pi, pj, ref = cache[kk]
        if tier == 2:
            assert by_pass_b(st, n, 2, pi, pj).any()
        elif W >= 8 and shape["variant"] == "smem":
            cz = compacts(st, n, W, kk, pi, pj)
            # whether any pair could skip compaction here: x's first group at least as large as y's, y0 = 1 .. n - 1
            y0 = np.arange(n)
            room = not compacts({"first_run": y0}, n, W, kk, y0, y0).all()
            assert cz.any(), f"W={W}: no pair compacts"
            assert (~cz).any() == room, f"W={W}: pairs that do not compact {(~cz).any()}, possible {room}"
        for persp in ("global", "local"):
            got = ik.run_pairs(x, (), perspective=persp, want_counts=True)
            assert_parity(got, ref[persp], f"n={n} tier {tier} W={W} {persp}")
    assert ran == list(range(1 if n <= 3000 else 3, 33))


@pytest.mark.parametrize("name", ["target", "config3", "config5", "config1", "config2"])
def test_benchmark_shapes_on_small_matrices(knobs, name):
    """bench.py's workloads run the many-units shape (W 16 kk 5 for the target); small matrices would plan the
    few-units one.  Forced to the benchmark's W, ten columns of each workload against the oracle."""
    x, persp = synth.make(name, C=10)
    n = x.shape[0]
    tier = tier_of(checked_stats(x), n)
    W = _lib.launch_shape(n, tier)["warps"]
    knobs(ICIKT_WARPS=W)
    assert _lib.launch_shape(n, tier)["warps"] == W
    if name == "target":
        assert (W, _lib.launch_shape(n, tier)["runs"], tier) == (16, 5, 0)
    check(x, persps=(persp, "local" if persp == "global" else "global"), what=f"{name} W={W}")


# ---------------------------------------------------------------- 5. register classes
@pytest.mark.parametrize("shape", ["cz", "plain", "gmem"])
def test_register_classes(knobs, shape):
    """ICIKT_REGCLASS 0 (64 registers), 1 (<512, 3>, 40) and 2 (<1024, 2>, 32) on a zero-compaction shape
    (n = 20 000, W 16), a shape without it (n = 3 000, W 2) and the global scratch (tier 2, pass B): the bytes of
    the unforced run, which matches the oracle."""
    if shape == "cz":
        x, W, env = synth.make("target", n=20000, C=8)[0], 16, dict(ICIKT_WARPS=16)
    elif shape == "plain":
        x, W, env = synth.make("config2", n=3000, C=8)[0], 2, dict(ICIKT_WARPS=2)
    else:
        x, W, env = tier2_matrix(4096, 17, 200, seed=21)[1], 32, dict(ICIKT_FORCE_GMEM=1)
    n, C = x.shape
    tier = tier_of(checked_stats(x), n)
    knobs(**env)
    assert _lib.launch_shape(n, tier)["warps"] == W
    assert _lib.launch_shape(n, tier)["variant"] == ("gmem" if shape == "gmem" else "smem")
    pi, pj = ordered_pairs(C)
    base = check(x, pi, pj, what=f"{shape} unforced")
    for cls in (0, 1, 2):
        knobs(ICIKT_REGCLASS=cls)
        for persp in ("global", "local"):
            got = ik.run_pairs(x, (), pi=pi, pj=pj, perspective=persp, want_counts=True)
            _same_pairs(got, base[persp], f"{shape} register class {cls} {persp}")
