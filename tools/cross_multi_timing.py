"""The cross calls over several GPUs (icikt_cross_pairs_multi / _edges_multi / _topk_multi) against one GPU.

Workloads:
1. Query against reference (the shape of r06_cross_timing.json): config-5 generator, 2 000 rows, Cx = 2 000 against
   Cy = 50 000 (10^8 pairs); the filtered call (|cor| >= 0.8) and the top-k call (k = 10, x side).
2. The target matrix (20 000 x 2 000, 25 % missing): icikt_cross_pairs of its first 1 000 columns against its last
   1 000 (10^6 pairs).
Arms: one GPU (the single-device call), devices = [0, 0] (the multi-device path on one GPU), and list(range(ndev))
when the box has more than one GPU.  Each arm is warmed up once and its result compared bit for bit with the one-GPU
result; then the arms alternate, `reps` runs each, and the medians are kept with the last run's timing parts.
The card's name, power limit, max SM clock and the device count come from the same run.

    python tools/cross_multi_timing.py [--reps 3] [--cy 50000] [--out r07_cross_multi_timing.json]
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


def card():
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True, check=True).stdout.strip()
    return dict(zip(q.split(","), (s.strip() for s in out.split(","))))


def med(v):
    return round(float(np.median(v)), 3)


def same(a, b):
    """bit for bit, arrays (float64 as int64) and nested dicts of them; timings are not results"""
    if isinstance(a, dict):
        return a.keys() == b.keys() and all(same(a[k], b[k]) for k in a if k != "timings")
    if isinstance(a, float):
        return np.float64(a).view(np.int64) == np.float64(b).view(np.int64)
    a, b = np.asarray(a), np.asarray(b)
    if a.dtype == np.float64:
        a, b = a.view(np.int64), b.view(np.int64)
    return a.shape == b.shape and np.array_equal(a, b)


def compare(call, arms, reps):
    """call(devices) -> result; the one-GPU arm is the reference"""
    ref = call(None)
    bit_identical = {name: bool(same(call(dev), ref)) for name, dev in arms.items() if dev is not None}
    runs = {name: [] for name in arms}
    last = {}
    for _ in range(reps):
        for name, dev in arms.items():
            t0 = time.perf_counter()
            r = call(dev)
            runs[name].append(1e3 * (time.perf_counter() - t0))
            last[name] = r["timings"]
    base = med(runs["one_gpu"])
    return dict(wall_ms={k: med(v) for k, v in runs.items()},
                speedup_vs_one_gpu={k: round(base / med(v), 3) for k, v in runs.items()},
                runs_ms={k: [round(x, 3) for x in v] for k, v in runs.items()},
                last_timings=last, bit_identical_to_one_gpu=bit_identical)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--cy", type=int, default=50000)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    ndev = _lib.load().icikt_device_count()
    if ndev < 1:
        raise SystemExit("no CUDA device")
    arms = {"one_gpu": None, "devices_0_0": [0, 0]}
    if ndev > 1:
        arms[f"devices_0_to_{ndev - 1}"] = list(range(ndev))
    res = dict(card=card(), device_count=ndev, arms={k: v for k, v in arms.items()}, reps=a.reps)

    n, cx, cy = 2000, 2000, a.cy
    x, _ = synth.make("config5", n=n, C=cx + cy)
    xa, ya = np.asfortranarray(x[:, :cx]), np.asfortranarray(x[:, cx:])
    del x
    q = dict(workload=f"config5 generator {n} rows: {cx} x {cy} = {cx * cy} pairs")
    q["edges |cor| >= 0.8"] = compare(lambda d: _lib.run_cross_edges(xa, ya, GLOBAL_NA, min_abs_cor=0.8, devices=d),
                                      arms, a.reps)
    q["topk k=10 x side"] = compare(lambda d: _lib.run_cross_topk(xa, ya, GLOBAL_NA, k=10, side="x", devices=d),
                                    arms, a.reps)
    res["query_reference"] = q
    del xa, ya

    x, _ = synth.make("target")
    C = x.shape[1]
    xa, ya = np.asfortranarray(x[:, :C // 2]), np.asfortranarray(x[:, C // 2:])
    t = dict(workload=f"target {x.shape[0]} x {C}: cross {C // 2} x {C - C // 2} = {(C // 2) * (C - C // 2)} pairs")
    t["pairs"] = compare(lambda d: _lib.run_cross(xa, ya, GLOBAL_NA, devices=d), arms, a.reps)
    res["target_cross_pairs"] = t

    s = json.dumps(res, indent=1)
    print(s)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(s + "\n")


if __name__ == "__main__":
    main()
