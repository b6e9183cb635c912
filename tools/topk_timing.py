"""The top-k all-pairs call (icikt_all_pairs_topk) against the filtered call (icikt_all_pairs_edges, t = 0.8) and
against K1 + sum of K2, on one GPU.

Workloads: config 5 (2 000 x 5 000 left-censored), 2 000 x 20 000 and, with --big, 2 000 x 60 000 left-censored;
k = 10 and 100.  The calls alternate after a warm-up; per call the wall time and the `timings` parts.  Both calls
walk the same windows and report K3 plus their selection as epilogue_ms, so the top-k selection's cost is
estimated as the top-k call's epilogue_ms minus the edges call's (whose selection is a compaction).  --profile
adds one torch.profiler run of the top-k call at 2 000 x 20 000, k = 100, with the device time of every kernel.
Config 5's lists are checked bit for bit against run_pairs sorted on the host.  The card's name, power limit and
max SM clock come from the same run.

    python tools/topk_timing.py [--reps 3] [--big] [--profile] [--out topk_timing.json]
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
T = 0.8
KS = (10, 100)


def card():
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True, check=True).stdout.strip()
    return dict(zip(q.split(","), (s.strip() for s in out.split(","))))


def timed(f, *a, **k):
    t0 = time.perf_counter()
    r = f(*a, **k)
    return 1e3 * (time.perf_counter() - t0), r


def check_lists(x, got, k):
    """config 5 only: the lists against run_pairs sorted per column on the host (abs order)"""
    full = _lib.run_pairs(x, GLOBAL_NA)
    C = x.shape[1]
    iu = np.triu_indices(C, 1)
    ok = full["status"] == 0
    pi, pj, raw = iu[0][ok], iu[1][ok], full["raw"][ok]
    col, partner, r = np.concatenate([pi, pj]), np.concatenate([pj, pi]), np.concatenate([raw, raw])
    order = np.lexsort((partner, -np.abs(r), col))
    col, partner, r = col[order], partner[order], r[order]
    rank = np.arange(col.size) - np.searchsorted(col, col)
    sel = rank < k
    idx = np.full((C, k), -1, dtype=np.int32)
    rw = np.full((C, k), np.nan)
    idx[col[sel], rank[sel]] = partner[sel]
    rw[col[sel], rank[sel]] = r[sel]
    assert np.array_equal(got["index"], idx) and np.array_equal(got["raw"].view(np.int64), rw.view(np.int64)), \
        "top-k lists differ from run_pairs sorted"


def summary(runs):
    keys = runs[0].keys()
    return dict(median={k: round(float(np.median([r[k] for r in runs])), 3) for k in keys},
                runs={k: [round(float(r[k]), 3) for r in runs] for k in keys})


def compare(name, x, reps, check=False):
    n, C = x.shape
    P = C * (C - 1) // 2
    for k in KS:  # warm-up of both calls and the cached plan
        _lib.run_topk(x, GLOBAL_NA, k=k)
    _lib.run_edges(x, GLOBAL_NA, min_abs_cor=T)
    arms = {f"topk_k{k}": [] for k in KS}
    arms["edges_t0.8"] = []
    for _ in range(reps):
        for k in KS:
            w, r = timed(_lib.run_topk, x, GLOBAL_NA, k=k)
            arms[f"topk_k{k}"].append(dict(wall_ms=w, **r["timings"]))
            if check and k == KS[0]:
                check_lists(x, r, k)
                check = False
            del r
        w, e = timed(_lib.run_edges, x, GLOBAL_NA, min_abs_cor=T)
        arms["edges_t0.8"].append(dict(wall_ms=w, **e["timings"]))
        kept = int(e["raw"].size)
        del e
    _lib.release_workspace()
    out = dict(workload=name, n=n, C=C, n_pairs=P, windows=-(-P // WINDOW), edges_rows_kept=kept,
               **{arm: summary(runs) for arm, runs in arms.items()})
    e = out["edges_t0.8"]["median"]
    k1_k2 = e["columns_ms"] + e["pairs_ms"]
    out["k1_plus_sum_k2_ms"] = round(k1_k2, 3)
    for k in KS:
        m = out[f"topk_k{k}"]["median"]
        sel = m["epilogue_ms"] - e["epilogue_ms"]
        out[f"topk_k{k}_vs"] = dict(wall_over_edges=round(m["wall_ms"] / e["wall_ms"], 4),
                                    wall_over_k1_k2=round(m["wall_ms"] / k1_k2, 4),
                                    selection_ms_est=round(sel, 3),
                                    selection_over_sum_k2=round(sel / m["pairs_ms"], 4))
    return out


def profile(x, k):
    import torch
    from torch.profiler import ProfilerActivity, profile as prof
    _lib.run_topk(x, GLOBAL_NA, k=k)
    with prof(activities=[ProfilerActivity.CUDA]) as p:
        _lib.run_topk(x, GLOBAL_NA, k=k)
        torch.cuda.synchronize()
    per = {}
    for ev in p.events():
        if ev.device_type == torch.autograd.DeviceType.CUDA:
            name = ev.name.split("(")[0].split("<")[0].split("::")[-1]
            a = per.setdefault(name, [0, 0.0])
            a[0] += 1
            a[1] += ev.device_time_total / 1e3
    _lib.release_workspace()
    return {name: dict(calls=c, ms=round(ms, 3)) for name, (c, ms) in sorted(per.items(), key=lambda kv: -kv[1][1])}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--big", action="store_true")
    ap.add_argument("--profile", action="store_true")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    info = card()
    print(json.dumps(info), flush=True)
    rows = []
    x, _ = synth.make("config5")
    rows.append(compare("config5 2000x5000", x, args.reps, check=True))
    print(json.dumps(rows[-1]), flush=True)
    x = synth.left_censored(2000, 20000, 0.20, seed=synth.SEEDS["config5"])
    rows.append(compare("2000x20000 left-censored", x, max(1, args.reps - 1)))
    print(json.dumps(rows[-1]), flush=True)
    prof_rows = None
    if args.profile:
        prof_rows = dict(workload="2000x20000 left-censored, top-k k=100", kernels=profile(x, 100))
        print(json.dumps(prof_rows), flush=True)
    del x
    if args.big:
        x = synth.left_censored(2000, 60000, 0.20, seed=synth.SEEDS["config5"])
        rows.append(compare("2000x60000 left-censored", x, 1))
        print(json.dumps(rows[-1]), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(dict(card=info, workloads=rows, profile=prof_rows), f, indent=1)


if __name__ == "__main__":
    main()
