"""The edge-count call (icikt_all_pairs_count_edges) at T = 1 and T = 64 filters against the filtered call
(icikt_all_pairs_edges) with the first filter, on one GPU.

Workloads: config 5 (2 000 x 5 000 left-censored) and C = 20 000 at n = 2 000.  Arms, alternating after a warm-up:
the filtered call at min_abs_cor = 0.8 without scale_max, the count at T = 1 with the same filter, the count at
T = 64 over thresholds 0.8 .. 0.99 (few pairs pass: the scattered degree atomics are rare) and at T = 64 over
0.0 .. 0.63 (most pairs pass most filters: one degree atomic per passing pair and filter).  Per call the wall time and
the `timings` parts: columns_ms is K1, pairs_ms the sum of K2 over the windows, epilogue_ms K3 with the selection or
the counting pass.  Every count at T = 1 is checked against the filtered call's row count.  The card's name, power
limit and max SM clock come from the same run.

    python tools/edge_count_timing.py [--reps 3] [--out edge_count_timing.json]
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

from icikendalltau_b200 import _lib, synth  # noqa: E402
from tools.edge_timing import GLOBAL_NA, WINDOW, card, summary, timed  # noqa: E402

T0 = 0.8
FEW = [(float(t), None) for t in np.linspace(0.8, 0.99, 64)]
MANY = [(float(t), None) for t in np.linspace(0.0, 0.63, 64)]


def compare(name, x, reps):
    n, C = x.shape
    P = C * (C - 1) // 2
    arms = {
        "edges_call": lambda: _lib.run_edges(x, GLOBAL_NA, min_abs_cor=T0, scale_max=False),
        "count_T1": lambda: _lib.run_count_edges(x, GLOBAL_NA, [(T0, None)]),
        "count_T64_few_pass": lambda: _lib.run_count_edges(x, GLOBAL_NA, FEW),
        "count_T64_most_pass": lambda: _lib.run_count_edges(x, GLOBAL_NA, MANY),
    }
    for f in arms.values():  # warm-up of every call and of the cached plans
        f()
    runs = {k: [] for k in arms}
    out = {}
    for _ in range(reps):
        for k, f in arms.items():
            w, r = timed(f)
            runs[k].append(dict(wall_ms=w, **r["timings"]))
            out[k] = r
    rows = int(out["edges_call"]["raw"].size)
    assert int(out["count_T1"]["n_pass"][0]) == rows, "T = 1 count differs from the filtered call's rows"
    assert int(out["count_T64_few_pass"]["n_pass"][0]) == rows
    _lib.release_workspace()
    return dict(workload=name, n=n, C=C, n_pairs=P, windows=-(-P // WINDOW), edges_rows=rows,
                passing_pairs_T64_few=int(out["count_T64_few_pass"]["n_pass"].sum()),
                passing_pairs_T64_most=int(out["count_T64_most_pass"]["n_pass"].sum()),
                **{k: summary(v) for k, v in runs.items()})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    info = card()
    print(json.dumps(info), flush=True)
    rows = []
    x, _ = synth.make("config5")
    rows.append(compare("config5 2000x5000", x, args.reps))
    print(json.dumps(rows[-1]), flush=True)
    x = synth.left_censored(2000, 20000, 0.20, seed=synth.SEEDS["config5"])
    rows.append(compare("2000x20000 left-censored", x, max(1, args.reps - 1)))
    print(json.dumps(rows[-1]), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(dict(card=info, workloads=rows), f, indent=1)


if __name__ == "__main__":
    main()
