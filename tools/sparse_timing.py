"""Sparse (CSC) input against its dense twin on one GPU: the one-shot all-pairs call (icikt_all_pairs_csc vs
icikt_all_pairs) on count data (config 4, 60 000 x 200, zeros = missing) and on a 20 000 x 2 000 left-censored
matrix at 10 % and 50 % density (present values stored, the rest dropped).  After a warm-up the two calls run
alternately; per workload it prints the wall time per call, the `timings` parts and the bytes sent to the device,
with the card's name and power limit from the same run.

    python tools/sparse_timing.py [--reps 3] [--out sparse_timing.json]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import scipy.sparse as sp

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


def workloads():
    x, _ = synth.make("config4")
    yield "config4 60000x200 counts", np.asfortranarray(np.nan_to_num(x, nan=0.0))
    for q in (0.9, 0.5):
        x = synth.left_censored(20000, 2000, q, seed=synth.SEEDS["target"])
        yield f"20000x2000 left-censored, density {1 - q:.0%}", np.asfortranarray(np.nan_to_num(x, nan=0.0))


def one_call(data):
    t0 = time.perf_counter()
    r = _lib.run_pairs(data, GLOBAL_NA)
    return time.perf_counter() - t0, r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    info = card()
    print(json.dumps(info), flush=True)
    rows = []
    for name, dense in workloads():
        a = sp.csc_matrix(dense)
        n, C = dense.shape
        bytes_dense = 8 * n * C
        bytes_csc = 8 * (C + 1) + 12 * a.nnz
        one_call(a)  # warm-up of both forms (and of the cached plan of this shape)
        one_call(dense)
        arms = {"sparse": [], "dense": []}
        for _ in range(args.reps):
            for arm, data in (("sparse", a), ("dense", dense)):
                wall, r = one_call(data)
                arms[arm].append(dict(wall_ms=1e3 * wall, **r["timings"]))
                if arm == "sparse":
                    last_sparse = r
                else:
                    assert np.array_equal(r["raw"].view(np.int64), last_sparse["raw"].view(np.int64)), name
        row = dict(workload=name, n=n, C=C, nnz=int(a.nnz), density=a.nnz / (n * C),
                   bytes_to_device=dict(sparse=bytes_csc, dense=bytes_dense))
        for arm, runs in arms.items():
            row[arm] = {k: [round(float(r[k]), 3) for r in runs] for k in runs[0]}
            row[arm]["median"] = {k: round(float(np.median([r[k] for r in runs])), 3) for k in runs[0]}
        rows.append(row)
        print(json.dumps(row), flush=True)
        _lib.release_workspace()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(dict(card=info, workloads=rows), f, indent=1)


if __name__ == "__main__":
    main()
