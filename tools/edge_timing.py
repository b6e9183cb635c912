"""The filtered all-pairs call (icikt_all_pairs_edges) against the per-pair call (icikt_all_pairs) on one GPU.

Workloads: config 5 (2 000 x 5 000 left-censored) and C = 20 000 at n = 2 000, the two calls alternating after a
warm-up; per call the wall time and the `timings` parts, and the filtered rows against run_pairs masked (bit for
bit).  --big adds C = 60 000 at n = 2 000, filtered call only (the per-pair call would need 68 B per pair on the
device): wall time, windows, rows kept and the bytes the per-pair and matrix calls would have needed.  The card's
name, power limit and max SM clock come from the same run.

    python tools/edge_timing.py [--reps 3] [--min-abs-cor 0.8] [--big] [--out edge_timing.json]
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

GLOBAL_NA = (np.nan, np.inf, 0.0)
WINDOW = 1 << 26  # the library's default ICIKT_EDGE_WINDOW


def card():
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True, check=True).stdout.strip()
    return dict(zip(q.split(","), (s.strip() for s in out.split(","))))


def timed(f, *a, **k):
    t0 = time.perf_counter()
    r = f(*a, **k)
    return 1e3 * (time.perf_counter() - t0), r


def check(edges, full, t):
    cor = full["raw"] / full["max_taumax"]
    idx = np.nonzero((full["status"] == 0) & (np.abs(cor) >= t))[0]
    ok = idx.size == edges["raw"].size and np.array_equal(edges["raw"].view(np.int64), full["raw"][idx].view(np.int64)) \
        and np.array_equal(edges["cor"].view(np.int64), cor[idx].view(np.int64))
    assert ok, "filtered rows differ from the per-pair result masked"


def summary(runs):
    keys = runs[0].keys()
    return dict(median={k: round(float(np.median([r[k] for r in runs])), 3) for k in keys},
                runs={k: [round(float(r[k]), 3) for r in runs] for k in keys})


def compare(name, x, t, reps):
    n, C = x.shape
    P = C * (C - 1) // 2
    _lib.run_edges(x, GLOBAL_NA, min_abs_cor=t)  # warm-up of both calls and their cached plans
    _lib.run_pairs(x, GLOBAL_NA)
    arms = {"filtered_call": [], "per_pair_call": []}
    kept = None
    for _ in range(reps):
        w, e = timed(_lib.run_edges, x, GLOBAL_NA, min_abs_cor=t)
        arms["filtered_call"].append(dict(wall_ms=w, **e["timings"]))
        kept = int(e["raw"].size)
        w, full = timed(_lib.run_pairs, x, GLOBAL_NA)
        arms["per_pair_call"].append(dict(wall_ms=w, **full["timings"]))
        check(e, full, t)
        del full
    _lib.release_workspace()
    return dict(workload=name, n=n, C=C, n_pairs=P, min_abs_cor=t, windows=-(-P // WINDOW), rows_kept=kept,
                **{arm: summary(runs) for arm, runs in arms.items()})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--min-abs-cor", type=float, default=0.8)
    ap.add_argument("--big", action="store_true")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    info = card()
    print(json.dumps(info), flush=True)
    t = args.min_abs_cor
    rows = []
    x, _ = synth.make("config5")
    rows.append(compare("config5 2000x5000", x, t, args.reps))
    print(json.dumps(rows[-1]), flush=True)
    x = synth.left_censored(2000, 20000, 0.20, seed=synth.SEEDS["config5"])
    rows.append(compare("2000x20000 left-censored", x, t, max(1, args.reps - 1)))
    print(json.dumps(rows[-1]), flush=True)
    del x
    if args.big:
        C = 60000
        x = synth.left_censored(2000, C, 0.20, seed=synth.SEEDS["config5"])
        P = C * (C - 1) // 2
        w, e = timed(_lib.run_edges, x, GLOBAL_NA, min_abs_cor=t, max_edges=400_000_000)
        _lib.release_workspace()
        rows.append(dict(workload="2000x60000 left-censored, filtered call only", n=2000, C=C, n_pairs=P,
                         min_abs_cor=t, windows=-(-P // WINDOW), rows_kept=int(e["raw"].size),
                         wall_ms=round(w, 1), timings={k: round(float(v), 3) for k, v in e["timings"].items()},
                         per_pair_call_bytes=dict(device=68 * P, host=36 * P),
                         matrix_call_bytes=dict(device=5 * 8 * C * C, host=5 * 8 * C * C),
                         rows_bytes_host=40 * int(e["raw"].size)))
        print(json.dumps(rows[-1]), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(dict(card=info, workloads=rows), f, indent=1)


if __name__ == "__main__":
    main()
