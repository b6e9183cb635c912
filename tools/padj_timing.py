"""The cost of adjusted p-values in the filtered all-pairs call, on one GPU.

Arms, alternating after a warm-up, on each input:
  plain   run_edges(max_pvalue = 0.05)                        the filtered call as before
  BH      run_edges(p_adjust = "BH", max_padj = 0.05)
  BY      run_edges(p_adjust = "BY", max_padj = 0.05)
  plain_cor  run_edges(min_abs_cor = 0.8)                     the baseline of BH_cor
  BH_cor  run_edges(p_adjust = "BH", min_abs_cor = 0.8)       max_padj NaN: every non-NaN p-value is a candidate
Inputs (n = 2 000, C = 20 000, 2 * 10^8 pairs, both seeded):
  left-censored   synth.left_censored(2000, 20000, 0.20), global_na = c(NA, Inf, 0)
  low-rank        one shared factor plus noise, so that nearly every pair has p <= 0.05 and the candidate buffer holds
                  ~2 * 10^8 keys
Reported per arm: median wall time and spread over `reps` runs, the last run's `timings`, rows and n_tests.  The
adjustment's device time (candidates, sort, scan, lookup) shows as the growth of epilogue_ms over its plain arm, and
BY's host sum of m terms as BY's wall time over BH's; the sum is also timed alone here with the same loop in NumPy
long double.  padj of BH and BY is checked bit for bit against oracle/p_adjust.py over run_pairs' p-values of the same
input.  The card's name, power limit and max SM clock come from the same run.

    python tools/padj_timing.py [--reps 3] [--out profiles/r09_padj_timing.json]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

from icikendalltau_b200 import _lib, synth  # noqa: E402
from oracle.p_adjust import by_q, p_adjust  # noqa: E402

GLOBAL_NA = (np.nan, np.inf, 0.0)
ARMS = {
    "plain": dict(max_pvalue=0.05),
    "BH": dict(p_adjust="BH", max_padj=0.05),
    "BY": dict(p_adjust="BY", max_padj=0.05),
    "plain_cor": dict(min_abs_cor=0.8),
    "BH_cor": dict(p_adjust="BH", min_abs_cor=0.8),
}


def card():
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True, check=True).stdout.strip()
    return dict(zip(q.split(","), (s.strip() for s in out.split(","))))


def low_rank(n, C, seed):
    rng = np.random.default_rng(seed)
    return np.asfortranarray(0.5 * rng.normal(size=(n, 1)) + rng.normal(size=(n, C)))


def check(x, gna, results):
    """padj of the BH and BY arms bit for bit against the oracle over run_pairs' p-values"""
    full = _lib.run_pairs(x, gna)
    pv = full["pvalue"]
    del full
    C = x.shape[1]
    out = {}
    for arm in ("BH", "BY"):
        r = results[arm]
        want = p_adjust(pv, arm)
        i, j = r["i"].astype(np.int64), r["j"].astype(np.int64)
        w = want[i * (2 * C - i - 1) // 2 + (j - i - 1)]  # the rows' positions in the combn order
        out[arm] = dict(rows=int(r["i"].size), n_tests=r["n_tests"],
                        oracle_rows=int((want <= 0.05).sum()),
                        bit_for_bit=bool(np.array_equal(w.view(np.int64), r["padj"].view(np.int64))
                                         and int((want <= 0.05).sum()) == r["i"].size))
    return out


def measure(name, x, gna, reps, do_check):
    for arm, kw in ARMS.items():  # warm-up of every arm
        _lib.run_edges(x, gna, **kw)
    times = {a: [] for a in ARMS}
    last = {}
    for _ in range(reps):
        for arm, kw in ARMS.items():
            t0 = time.perf_counter()
            r = _lib.run_edges(x, gna, **kw)
            times[arm].append(time.perf_counter() - t0)
            last[arm] = r
    row = dict(input=name, arms={})
    for arm in ARMS:
        r = last[arm]
        v = np.array(times[arm])
        row["arms"][arm] = dict(median_s=round(float(np.median(v)), 4), min_s=round(float(v.min()), 4),
                                max_s=round(float(v.max()), 4), rows=int(r["i"].size), n_tests=r.get("n_tests"),
                                timings=r["timings"])
    a = row["arms"]
    base = {"BH": "plain", "BY": "plain", "BH_cor": "plain_cor"}
    row["epilogue_growth_ms"] = {k: round(a[k]["timings"]["epilogue_ms"] - a[b]["timings"]["epilogue_ms"], 2)
                                 for k, b in base.items()}
    row["overhead_vs_plain"] = {k: round(a[k]["median_s"] / a[b]["median_s"], 4) for k, b in base.items()}
    row["by_minus_bh_s"] = round(a["BY"]["median_s"] - a["BH"]["median_s"], 4)
    m = a["BH"]["n_tests"]
    t0 = time.perf_counter()
    by_q(m)
    row["by_sum_numpy_longdouble_s"] = round(time.perf_counter() - t0, 3)
    if do_check:
        row["check"] = check(x, gna, last)
    print(json.dumps(row), flush=True)
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--C", type=int, default=20000)
    ap.add_argument("--no-check", action="store_true")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r09_padj_timing.json"))
    args = ap.parse_args()
    rec = dict(card=card(), reps=args.reps, arms=ARMS, rows=[])
    x = synth.left_censored(2000, args.C, 0.20, seed=synth.SEEDS["config5"])
    rec["rows"].append(measure(f"2000x{args.C} left-censored", x, GLOBAL_NA, args.reps, not args.no_check))
    del x
    x = low_rank(2000, args.C, seed=synth.SEEDS["config5"])
    rec["rows"].append(measure(f"2000x{args.C} low-rank", x, (), args.reps, not args.no_check))
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(rec, f, indent=1)


if __name__ == "__main__":
    main()
