"""Pair-kernel time (K2, the `pairs_ms` part of a one-shot all-pairs call) of two builds of libicikt_b200.so,
alternating, on one GPU, for a synthetic matrix of any shape: n rows x C columns, a fraction q of every column
left-censored (missing), tie-free values.  q = 0 gives columns without missing values, where leaving the
lowest-rank keys out of pass A saves nothing and only its cost shows.  Prints the card's name, power limit and
max SM clock, then one JSON line per run and the median per build.

    python tools/k2_ab_timing.py --lib-a OLD.so --lib-b NEW.so --n 20000 --cols 400 --q 0 --reps 3
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

ONE = r"""
import json, sys
import numpy as np
sys.path.insert(0, sys.argv[1])
import icikendalltau_b200 as ik
from icikendalltau_b200 import synth
n, C, q, steps = int(sys.argv[2]), int(sys.argv[3]), float(sys.argv[4]), int(sys.argv[5])
x = synth.left_censored(n, C, q, 7) if q > 0 else np.asfortranarray(np.random.default_rng(7).standard_normal((n, C)))
ik.run_pairs(x, ())  # warm-up: module load, workspace
ms = [ik.run_pairs(x, ())["timings"]["pairs_ms"] for _ in range(steps)]
print(json.dumps({"pairs_ms": sorted(ms)[len(ms) // 2], "all": ms}))
"""


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib-a", required=True)
    ap.add_argument("--lib-b", required=True)
    ap.add_argument("--n", type=int, default=20000)
    ap.add_argument("--cols", type=int, default=400)
    ap.add_argument("--q", type=float, default=0.0)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--steps", type=int, default=3)
    a = ap.parse_args()
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip()
    print(json.dumps({"card": card, "n": a.n, "cols": a.cols, "q": a.q}), flush=True)
    res = {"a": [], "b": []}
    for r in range(a.reps):
        for arm, lib in (("a", a.lib_a), ("b", a.lib_b)):
            env = dict(os.environ, ICIKT_LIB_PATH=os.path.abspath(lib))
            out = subprocess.run([sys.executable, "-c", ONE, ROOT, str(a.n), str(a.cols), str(a.q), str(a.steps)],
                                 env=env, capture_output=True, text=True, check=True).stdout.strip().splitlines()[-1]
            d = json.loads(out)
            res[arm].append(d["pairs_ms"])
            print(json.dumps({"arm": arm, "rep": r, **d}), flush=True)
    med = {k: sorted(v)[len(v) // 2] for k, v in res.items()}
    print(json.dumps({"median_pairs_ms": med, "b_over_a": med["b"] / med["a"]}), flush=True)


if __name__ == "__main__":
    main()
