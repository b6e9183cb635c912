"""The cross calls (icikt_cross_pairs / _edges / _topk) on one GPU.

1. The target matrix (20 000 x 2 000, 25 % missing, global perspective): icikt_cross_pairs of its first 1 000 columns
   against its last 1 000 (10^6 pairs) against icikt_pair_list on the same 10^6 pairs of the whole matrix
   (pi = i, pj = 1 000 + j), alternating after a warm-up; the two results are compared bit for bit.  Beside them,
   icikt_all_pairs on the whole matrix (1 999 000 pairs): the per-pair work is the same, so the pair rates should be
   close.
2. Query against reference at n = 2 000: Cx = 2 000 against Cy = 50 000 (10^8 pairs), the filtered call (|cor| >= 0.8)
   and the top-k call (k = 10, x side only), with the device memory in use before and during each call
   (cudaMemGetInfo through torch.cuda.mem_get_info, sampled by a thread every 20 ms).
The card's name, power limit and max SM clock come from the same run.

    python tools/cross_timing.py [--reps 3] [--cy 50000] [--out cross_timing.json]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

from icikendalltau_b200 import _lib, synth  # noqa: E402

GLOBAL_NA = (np.nan, np.inf, 0.0)


def card():
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True, check=True).stdout.strip()
    return dict(zip(q.split(","), (s.strip() for s in out.split(","))))


def timed(f, *a, **k):
    t0 = time.perf_counter()
    r = f(*a, **k)
    return 1e3 * (time.perf_counter() - t0), r


class PeakMemory:
    """device memory in use (total - free, cudaMemGetInfo) before the call and its peak while the call runs"""

    def __init__(self):
        import torch
        self.info = lambda: torch.cuda.mem_get_info(0)

    def __enter__(self):
        free, total = self.info()
        self.before = total - free
        self.peak = self.before
        self.stop = False
        self.th = threading.Thread(target=self._poll, daemon=True)
        self.th.start()
        return self

    def _poll(self):
        while not self.stop:
            free, total = self.info()
            self.peak = max(self.peak, total - free)
            time.sleep(0.02)

    def __exit__(self, *exc):
        self.stop = True
        self.th.join()
        free, total = self.info()
        self.peak = max(self.peak, total - free)

    def as_dict(self):
        return dict(before_gb=round(self.before / 1e9, 3), peak_gb=round(self.peak / 1e9, 3),
                    added_gb=round((self.peak - self.before) / 1e9, 3))


def med(v):
    return round(float(np.median(v)), 3)


def target_part(reps):
    x, _ = synth.make("target")
    n, C = x.shape
    cx = C // 2
    xa, ya = np.asfortranarray(x[:, :cx]), np.asfortranarray(x[:, cx:])
    P = cx * (C - cx)
    p = np.arange(P)
    pi, pj = (p // (C - cx)).astype(np.int32), (cx + p % (C - cx)).astype(np.int32)
    # warm-up (cached plans, module loads), then the bit-for-bit check
    cross = _lib.run_cross(xa, ya, GLOBAL_NA)
    plist = _lib.run_pairs(x, GLOBAL_NA, pi=pi, pj=pj)
    for k in ("raw", "pvalue", "taumax", "completeness"):
        assert np.array_equal(cross[k].view(np.int64), plist[k].view(np.int64)), f"cross vs pair list: {k}"
    assert np.array_equal(cross["status"], plist["status"])
    _lib.run_pairs(x, GLOBAL_NA)
    t = dict(cross=[], pair_list=[], all_pairs=[], cross_pairs_ms=[], pair_list_pairs_ms=[], all_pairs_pairs_ms=[])
    for _ in range(reps):
        ms, r = timed(_lib.run_cross, xa, ya, GLOBAL_NA)
        t["cross"].append(ms)
        t["cross_pairs_ms"].append(r["timings"]["pairs_ms"])
        ms, r = timed(_lib.run_pairs, x, GLOBAL_NA, pi=pi, pj=pj)
        t["pair_list"].append(ms)
        t["pair_list_pairs_ms"].append(r["timings"]["pairs_ms"])
        ms, r = timed(_lib.run_pairs, x, GLOBAL_NA)
        t["all_pairs"].append(ms)
        t["all_pairs_pairs_ms"].append(r["timings"]["pairs_ms"])
    P_all = C * (C - 1) // 2
    return dict(workload=f"target {n} x {C}: cross {cx} x {C - cx} = {P} pairs; all pairs {P_all}",
                wall_ms=dict(cross=med(t["cross"]), pair_list=med(t["pair_list"]), all_pairs=med(t["all_pairs"])),
                k2_ms=dict(cross=med(t["cross_pairs_ms"]), pair_list=med(t["pair_list_pairs_ms"]),
                           all_pairs=med(t["all_pairs_pairs_ms"])),
                pairs_per_s_wall=dict(cross=round(P / (med(t["cross"]) / 1e3)),
                                      pair_list=round(P / (med(t["pair_list"]) / 1e3)),
                                      all_pairs=round(P_all / (med(t["all_pairs"]) / 1e3))),
                runs_ms={k: [round(v, 3) for v in vals] for k, vals in t.items()},
                last_cross_timings=cross["timings"], bit_identical_to_pair_list=True)


def query_part(reps, cy):
    n, cx = 2000, 2000
    x, _ = synth.make("config5", n=n, C=cx + cy)
    xa, ya = np.asfortranarray(x[:, :cx]), np.asfortranarray(x[:, cx:])
    del x
    out = dict(workload=f"config5 generator {n} rows: {cx} x {cy} = {cx * cy} pairs")
    _lib.run_cross_topk(xa, ya[:, :1000], GLOBAL_NA, k=10, side="x")  # module loads
    for name, f, kw in (("edges |cor| >= 0.8", _lib.run_cross_edges, dict(min_abs_cor=0.8)),
                        ("topk k=10 x side", _lib.run_cross_topk, dict(k=10, side="x"))):
        _lib.release_workspace()
        runs, mem, tms = [], None, None
        for r in range(reps):
            if r == 0:
                with PeakMemory() as pm:
                    ms, res = timed(f, xa, ya, GLOBAL_NA, **kw)
                mem = pm.as_dict()
            else:
                ms, res = timed(f, xa, ya, GLOBAL_NA, **kw)
            runs.append(ms)
            tms = res["timings"]
        rows = int(res["i"].size) if "i" in res else int(res["x_side"]["n_neighbors"].sum())
        out[name] = dict(wall_ms=med(runs), runs_ms=[round(v, 3) for v in runs], pairs_per_s=round(cx * cy / (med(runs) / 1e3)),
                         first_call_device_memory=mem, rows_or_entries=rows, timings=tms)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--cy", type=int, default=50000)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    res = dict(card=card(), target=target_part(a.reps), query_reference=query_part(a.reps, a.cy))
    s = json.dumps(res, indent=1)
    print(s)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(s + "\n")


if __name__ == "__main__":
    main()
