"""The filtered and top-k all-pairs calls over several GPUs of one box (icikt_all_pairs_edges_multi,
icikt_all_pairs_topk_multi) against the same calls on one GPU.

Workloads: 2 000 x 20 000 left-censored (and, with --big, 2 000 x 60 000), global_na = c(NA, Inf, 0); edges at
min_abs_cor = 0.8 with scale_max, top-k with k = 10 and 100.  Arms: 1, 2, 4 and 8 GPUs, as many as the box has;
--repeat adds [0, 0] (the multi-device path on one GPU: what the slicing and the merge cost without more hardware).
After a warm-up of every arm the arms alternate; per arm the median and the spread of the wall time and the `timings`
parts the call returns (the slowest device's figures, n_launches summed).  Every multi-device result is checked bit
for bit against the one-GPU result.  The card's name, power limit and max SM clock come from the same run.

    python tools/window_multi_timing.py [--reps 3] [--big] [--repeat] [--out profiles/window_multi_timing.json]
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
T = 0.8


def cards():
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()
    return [dict(zip(q.split(","), (s.strip() for s in line.split(",")))) for line in out]


def timed(f, *a, **k):
    t0 = time.perf_counter()
    r = f(*a, **k)
    return 1e3 * (time.perf_counter() - t0), r


def same(a, b, keys):
    for k in keys:
        x, y = np.asarray(a[k]), np.asarray(b[k])
        assert x.shape == y.shape and np.array_equal(x.view(np.uint8), y.view(np.uint8)), k
    assert np.float64(a["max_taumax"]).tobytes() == np.float64(b["max_taumax"]).tobytes()


def summary(runs):
    keys = runs[0].keys()
    med = {k: round(float(np.median([r[k] for r in runs])), 3) for k in keys}
    spread = {k: round(float(max(r[k] for r in runs) - min(r[k] for r in runs)), 3) for k in keys}
    return dict(median=med, spread=spread, runs={k: [round(float(r[k]), 3) for r in runs] for k in keys})


def measure(name, x, arms, reps, warm):
    n, C = x.shape
    calls = {"edges": (lambda dev: _lib.run_edges(x, GLOBAL_NA, min_abs_cor=T, devices=dev),
                       ("i", "j", "cor", "raw", "pvalue", "taumax", "completeness")),
             "topk10": (lambda dev: _lib.run_topk(x, GLOBAL_NA, k=10, devices=dev),
                        ("index", "n_neighbors", "cor", "raw", "pvalue", "taumax", "completeness")),
             "topk100": (lambda dev: _lib.run_topk(x, GLOBAL_NA, k=100, devices=dev),
                         ("index", "n_neighbors", "cor", "raw", "pvalue", "taumax", "completeness"))}
    out = []
    for call, (f, keys) in calls.items():
        ref = None
        if warm:
            for label, dev in arms:
                r = f(dev)
                ref = ref or r
                same(r, ref, keys)
        runs = {label: [] for label, _ in arms}
        for _ in range(reps):
            for label, dev in arms:
                w, r = timed(f, dev)
                runs[label].append(dict(wall_ms=w, **r["timings"]))
                ref = ref or r
                same(r, ref, keys)
        rows = int(ref["raw"].size) if call == "edges" else None
        del ref
        row = dict(workload=name, call=call, n=n, C=C, n_pairs=C * (C - 1) // 2, rows_kept=rows, bit_for_bit=True,
                   arms={label: summary(v) for label, v in runs.items()})
        print(json.dumps(row), flush=True)
        out.append(row)
        _lib.release_workspace()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--big", action="store_true")
    ap.add_argument("--repeat", action="store_true")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    info = cards()
    print(json.dumps(info), flush=True)
    ndev = _lib.load().icikt_device_count()
    arms = [("1 GPU", None)] + [(f"{g} GPUs", list(range(g))) for g in (2, 4, 8) if g <= ndev]
    if args.repeat:
        arms.append(("[0, 0]", [0, 0]))
    rows = []
    x = synth.left_censored(2000, 20000, 0.20, seed=synth.SEEDS["config5"])
    rows += measure("2000x20000 left-censored", x, arms, args.reps, warm=True)
    del x
    if args.big:
        x = synth.left_censored(2000, 60000, 0.20, seed=synth.SEEDS["config5"])
        rows += measure("2000x60000 left-censored", x, arms, max(1, args.reps - 2), warm=False)
        del x
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(dict(cards=info, device_count=ndev, min_abs_cor=T, workloads=rows), f, indent=1)


if __name__ == "__main__":
    main()
