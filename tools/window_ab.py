"""The windowed calls of two builds of libicikt_b200.so, alternating in fresh processes on one GPU: outputs and speed.

Calls: run_edges (|cor| >= 0.8, scale_max), run_topk (k = 10 and 100), run_cross, run_cross_edges (|cor| >= 0.8) and
run_cross_topk (k = 10, side "both"), each on dense and on CSC input (NaN -> 0, an implicit zero; global_na =
c(NA, Inf, 0) makes both forms the same data), on one GPU (the single-device entry point) and on devices = [0, 0] (the
multi-device entry point, two workers on one GPU).  Sizes: 2 000 x 20 000 left-censored (synth.left_censored, 20 %
missing) for the all-pairs calls; 2 000 queries x 20 000 references of the same generator (n = 2 000) for the cross
calls; and 200 x 50 (cross: 200 x 50 against 200 x 50), where the per-call host overhead dominates.

Each worker process loads one build (ICIKT_LIB_PATH), and per case makes one warm-up call, then --steps timed calls
back to back (--small-steps at the small size).  The builds alternate over --reps rounds (a b, then b a, ...).  Per
case and build: the median wall time and its spread (min, max) over every timed call, the median of every `timings`
field, and a hash of every output array.  Every output must be bit-identical between the builds, and each build's
median must lie within the other build's spread.  The card's name, power limit and max SM clock come from the same
run.

--calls pairs runs the per-pair and matrix calls instead: run_pairs over all pairs at the benchmark's target (the
pipelined call on one GPU; 200 x 50 at the small size), run_pairs with a list of 10^5 random pairs of that matrix (500
at the small size, one GPU only), and run_matrices (diag_good) at 2 000 x 5 000 (200 x 50), each dense and CSC, on one
GPU and, where the call takes devices, on devices = [0, 0].

    python tools/window_ab.py --lib-a OLD.so --lib-b NEW.so [--calls windowed|pairs] [--reps 2] [--steps 3]
                              [--sizes big,small] [--only TEXT] [--out f.json]

--only keeps the cases whose name contains TEXT (e.g. "cross big": the per-pair cross call at the large size).
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.dont_write_bytecode = True
GLOBAL_NA = (np.nan, np.inf, 0.0)
T = 0.8


def card():
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()
    return [dict(zip(q.split(","), (s.strip() for s in line.split(",")))) for line in out]


def digest(r):
    """a hash of every output array (nested dicts of the cross top-k call included) and of max_taumax"""
    out = {}
    for k, v in sorted(r.items()):
        if k == "timings":
            continue
        if isinstance(v, dict):
            out.update({f"{k}.{kk}": vv for kk, vv in digest(v).items()})
        else:
            out[k] = hashlib.blake2b(np.ascontiguousarray(v).tobytes(), digest_size=16).hexdigest()
    return out


def cases(sizes):
    """(name, call) for every case, grouped so that consecutive cases reuse the cached window plans"""
    import scipy.sparse as sp
    from icikendalltau_b200 import _lib, synth

    def forms(a):
        return {"dense": a, "csc": sp.csc_matrix(np.nan_to_num(a, nan=0.0))}

    for size in sizes:
        if size == "big":
            n, C, cx, cy = 2000, 20000, 2000, 20000
        else:
            n, C, cx, cy = 200, 50, 50, 50
        x = synth.left_censored(n, C, 0.20, seed=synth.SEEDS["config5"])
        for form, data in forms(x).items():
            for arm, dev in (("one_gpu", None), ("devices_0_0", [0, 0])):
                tag = f"{size} {n}x{C} {form} {arm}"
                yield f"edges {tag}", lambda d=data, v=dev: _lib.run_edges(d, GLOBAL_NA, min_abs_cor=T, devices=v)
                for k in (10, 100):
                    yield f"topk{k} {tag}", lambda d=data, v=dev, k=k: _lib.run_topk(d, GLOBAL_NA, k=k, devices=v)
        del x
        xy = synth.left_censored(n, cx + cy, 0.20, seed=synth.SEEDS["config5"])
        xs, ys = forms(np.asfortranarray(xy[:, :cx])), forms(np.asfortranarray(xy[:, cx:]))
        del xy
        for form in ("dense", "csc"):
            xa, ya = xs[form], ys[form]
            for arm, dev in (("one_gpu", None), ("devices_0_0", [0, 0])):
                tag = f"{size} {n}: {cx}x{cy} {form} {arm}"
                yield f"cross {tag}", lambda a=xa, b=ya, v=dev: _lib.run_cross(a, b, GLOBAL_NA, devices=v)
                yield f"cross_edges {tag}", lambda a=xa, b=ya, v=dev: _lib.run_cross_edges(a, b, GLOBAL_NA, min_abs_cor=T,
                                                                                         devices=v)
                yield f"cross_topk10 {tag}", lambda a=xa, b=ya, v=dev: _lib.run_cross_topk(a, b, GLOBAL_NA, k=10,
                                                                                          side="both", devices=v)


def pair_cases(sizes):
    """(name, call) for the per-pair and matrix calls: run_pairs over all pairs (at the benchmark's target, the
    pipelined call on one GPU), run_pairs with a pair list, and run_matrices (all pairs, diag_good)"""
    import scipy.sparse as sp
    from icikendalltau_b200 import _lib, synth

    def forms(a):
        return {"dense": a, "csc": sp.csc_matrix(np.nan_to_num(a, nan=0.0))}

    arms = (("one_gpu", None), ("devices_0_0", [0, 0]))
    for size in sizes:
        if size == "big":
            x, _ = synth.make("target")
            P, (mn, mc) = 100_000, (2000, 5000)
        else:
            x = synth.left_censored(200, 50, 0.20, seed=synth.SEEDS["config5"])
            P, (mn, mc) = 500, (200, 50)
        n, C = x.shape
        rng = np.random.default_rng(5)
        pi, pj = rng.integers(0, C, P).astype(np.int32), rng.integers(0, C, P).astype(np.int32)
        for form, data in forms(x).items():
            tag = f"{size} {n}x{C} {form}"
            yield f"pair_list {tag} P={P} one_gpu", lambda d=data: _lib.run_pairs(d, GLOBAL_NA, pi=pi, pj=pj)
            for arm, dev in arms:
                yield f"pairs {tag} {arm}", lambda d=data, v=dev: _lib.run_pairs(d, GLOBAL_NA, devices=v)
        del x, data
        m = synth.left_censored(mn, mc, 0.20, seed=synth.SEEDS["config5"])
        for form, data in forms(m).items():
            for arm, dev in arms:
                yield f"matrices {size} {mn}x{mc} {form} {arm}", lambda d=data, v=dev: _lib.run_matrices(d, GLOBAL_NA,
                                                                                                        devices=v)


def worker(a):
    """one process, one build: every case once for warm-up, then its timed calls; one JSON document on stdout"""
    sys.path.insert(0, ROOT)
    res = {}
    sizes = a.sizes.split(",")
    for name, call in (pair_cases(sizes) if a.calls == "pairs" else cases(sizes)):
        if a.only not in name:
            continue
        call()
        steps = a.steps if name.split()[1] == "big" else a.small_steps
        wall, tms = [], []
        for _ in range(steps):
            t0 = time.perf_counter()
            r = call()
            wall.append(1e3 * (time.perf_counter() - t0))
            tms.append(r["timings"])
        res[name] = dict(wall_ms=wall, timings=tms, hashes=digest(r))
        del r
    print(json.dumps(res))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib-a")
    ap.add_argument("--lib-b")
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--small-steps", type=int, default=30)
    ap.add_argument("--sizes", default="big,small")
    ap.add_argument("--only", default="")
    ap.add_argument("--calls", choices=("windowed", "pairs"), default="windowed")
    ap.add_argument("--out", default=None)
    ap.add_argument("--worker", action="store_true")
    a = ap.parse_args()
    if a.worker:
        return worker(a)
    libs = {"a": os.path.abspath(a.lib_a), "b": os.path.abspath(a.lib_b)}
    res = dict(card=card(), libs=libs, reps=a.reps, steps=a.steps, small_steps=a.small_steps, only=a.only,
               calls=a.calls, cases={})
    print(json.dumps(res["card"]), flush=True)
    runs = {"a": [], "b": []}
    for rep in range(a.reps):
        for arm in ("a", "b") if rep % 2 == 0 else ("b", "a"):
            t0 = time.perf_counter()
            cmd = [sys.executable, os.path.abspath(__file__), "--worker", "--steps", str(a.steps),
                   "--small-steps", str(a.small_steps), "--sizes", a.sizes, "--only", a.only, "--calls", a.calls]
            out = subprocess.run(cmd, env=dict(os.environ, ICIKT_LIB_PATH=libs[arm]), capture_output=True, text=True)
            if out.returncode:
                sys.stderr.write(out.stderr)
                raise SystemExit(f"worker of build {arm} failed")
            runs[arm].append(json.loads(out.stdout.strip().splitlines()[-1]))
            print(json.dumps({"rep": rep, "build": arm, "s": round(time.perf_counter() - t0, 1)}), flush=True)
    ok = True
    for name in runs["a"][0]:
        c = {}
        for arm in ("a", "b"):
            wall = [w for r in runs[arm] for w in r[name]["wall_ms"]]
            tms = [t for r in runs[arm] for t in r[name]["timings"]]
            c[arm] = dict(median_ms=round(float(np.median(wall)), 3), min_ms=round(min(wall), 3),
                          max_ms=round(max(wall), 3), wall_ms=[round(w, 3) for w in wall],
                          timings={k: round(float(np.median([t[k] for t in tms])), 3) for k in tms[0]})
        hashes = [r[name]["hashes"] for arm in ("a", "b") for r in runs[arm]]
        c["hashes"] = hashes[0]
        c["identical"] = all(h == hashes[0] for h in hashes)
        c["within_spread"] = (c["b"]["min_ms"] <= c["a"]["median_ms"] <= c["b"]["max_ms"]
                              and c["a"]["min_ms"] <= c["b"]["median_ms"] <= c["a"]["max_ms"])
        c["b_over_a"] = round(c["b"]["median_ms"] / c["a"]["median_ms"], 4)
        ok = ok and c["identical"]
        res["cases"][name] = c
        print(f"{name:48s} a {c['a']['median_ms']:10.3f} [{c['a']['min_ms']:.3f}, {c['a']['max_ms']:.3f}]  "
              f"b {c['b']['median_ms']:10.3f} [{c['b']['min_ms']:.3f}, {c['b']['max_ms']:.3f}]  "
              f"b/a {c['b_over_a']:.4f}  identical {c['identical']}  within {c['within_spread']}", flush=True)
    res["all_identical"] = ok
    res["all_within_spread"] = all(c["within_spread"] for c in res["cases"].values())
    print(json.dumps({"all_identical": ok, "all_within_spread": res["all_within_spread"]}), flush=True)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(json.dumps(res, indent=1) + "\n")
    if not ok:
        raise SystemExit("outputs differ between the builds")


if __name__ == "__main__":
    main()
