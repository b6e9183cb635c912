"""The component call (icikt_all_pairs_components) against the edge-count call (icikt_all_pairs_count_edges) on the
same filters, on one GPU.

Workloads: config 5 (2 000 x 5 000 left-censored), 2 000 x 20 000 left-censored, and 2 000 x 20 000 with planted
sample groups (8 groups, each column its group's signal plus noise of the same variance: |tau| about 1/3 within a
group, about 0 across), where many components survive across the grid while a large share of the pairs pass.  Filter
sets: T = 1 at min_abs_cor = 0.8; T = 64 over 0.8 .. 0.99 (few pairs pass); T = 64 over 0.0 .. 0.63 (most pairs pass
most filters); on the planted matrix, T = 64 over 0.0 .. 0.63 as well.  Each count call and the components call on
the same filters alternate after a warm-up.  Per call the wall time and the `timings` parts: pairs_ms is the sum of
K2, epilogue_ms K3 with the counting pass (and the unions), d2h_ms the labels kernel and the copy out.  The counts of
the two calls are checked equal.  The card's name, power limit and max SM clock come from the same run.

    python tools/component_timing.py [--reps 3] [--out component_timing.json]
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

T1 = [(0.8, None)]
FEW = [(float(t), None) for t in np.linspace(0.8, 0.99, 64)]
MANY = [(float(t), None) for t in np.linspace(0.0, 0.63, 64)]


def planted(n, C, groups, seed):
    rng = np.random.default_rng(seed)
    g = rng.integers(0, groups, C)
    base = rng.normal(size=(n, groups))
    return np.asfortranarray(base[:, g] + rng.normal(size=(n, C)))


def compare(name, x, sets, reps):
    n, C = x.shape
    P = C * (C - 1) // 2
    arms = {}
    for sname, f in sets.items():
        arms[f"count_{sname}"] = lambda f=f: _lib.run_count_edges(x, GLOBAL_NA, f)
        arms[f"components_{sname}"] = lambda f=f: _lib.run_count_edges(x, GLOBAL_NA, f, want_components=True)
    for f in arms.values():  # warm-up of every call and of the cached plans
        f()
    runs = {k: [] for k in arms}
    out = {}
    for _ in range(reps):
        for k, f in arms.items():
            w, r = timed(f)
            runs[k].append(dict(wall_ms=w, **r["timings"]))
            out[k] = r
    row = dict(workload=name, n=n, C=C, n_pairs=P, windows=-(-P // WINDOW))
    for sname in sets:
        c, k = out[f"count_{sname}"], out[f"components_{sname}"]
        for key in ("n_pass", "degree", "status_counts"):
            assert np.array_equal(c[key], k[key]), (sname, key)
        ms = lambda a: float(np.median([r["wall_ms"] for r in runs[a]]))  # noqa: E731
        row[sname] = dict(T=len(sets[sname]), passing_pairs=int(c["n_pass"].sum()),
                          filters_one_component=int((k["n_components"] == 1).sum()),
                          n_components=k["n_components"].tolist(),
                          count=summary(runs[f"count_{sname}"]), components=summary(runs[f"components_{sname}"]),
                          wall_change_pct=100.0 * (ms(f"components_{sname}") / ms(f"count_{sname}") - 1.0))
    _lib.release_workspace()
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    info = card()
    print(json.dumps(info), flush=True)
    rows = []
    sets = dict(T1=T1, T64_few_pass=FEW, T64_most_pass=MANY)
    x, _ = synth.make("config5")
    rows.append(compare("config5 2000x5000", x, sets, args.reps))
    print(json.dumps(rows[-1]), flush=True)
    x = synth.left_censored(2000, 20000, 0.20, seed=synth.SEEDS["config5"])
    rows.append(compare("2000x20000 left-censored", x, sets, max(1, args.reps - 1)))
    print(json.dumps(rows[-1]), flush=True)
    x = planted(2000, 20000, 8, seed=12)
    rows.append(compare("2000x20000 planted 8 groups", x, dict(T64_planted=MANY), max(1, args.reps - 1)))
    print(json.dumps(rows[-1]), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(dict(card=info, workloads=rows), f, indent=1)


if __name__ == "__main__":
    main()
