#!/usr/bin/env python
"""bench.py -- column-pairs/sec of the all-pairs ICI-Kendall-tau hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W]
                    [--workload target|config1|config2|config3|config4|config5]
                    [--impl b200|reference] [--scaling strong|weak] [--dump-outputs DIR]

Default workload: the north-star TARGET (2 000 samples x 20 000 features, 25 % left-censored,
1 999 000 pairs), which fits one GPU.  N > 1 (torchrun, one rank per GPU) defaults to STRONG scaling
of that same matrix: every rank uploads and preprocesses (K1) its slice of the columns, the ranks
all-gather the per-column tables over NCCL/NVLink, and every rank computes one contiguous slice of
the pair order (K2 + K3) -- no collective on the pair path itself.  `--scaling weak` keeps the pairs
per GPU constant instead by growing the number of samples with sqrt(N).

A step = one pass of the hot path (K1 + table exchange + K2 + K3) over one synthetic left-censored
matrix (icikendalltau_b200/synth.py).  `value` is measured with the matrix resident in HBM; `e2e` is
the same metric from HOST buffers to HOST results (pinned input; H2D and D2H inside the timed
region) through the public call -- the one-shot C ABI `icikt_all_pairs` at N = 1, the plan API under
torchrun; `e2e_pageable` repeats it from a plain NumPy array into freshly allocated outputs, which is
what an R caller hands over.  After the timed region a seeded sample of pairs is checked against the
CPU oracle (`parity_sample`).

--dump-outputs DIR writes what the timed plan returned for its last step as DIR/<name>.npy (see
dump_outputs).  The inputs are seeded, so two builds run with the same arguments can be compared
array for array.

--impl reference times the reference's CPU path.  R and Rcpp are not installed in this image, so
the true Rcpp+furrr path cannot run; the arm times the line-faithful C++ restatement (oracle/,
`kind: port`) with one thread per contiguous chunk like furrr's workers.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark leaves the tree as it found it (it may be read-only)

METRIC = "column-pairs/sec"
P_TOL = 1e-12  # p-value: |dp| <= P_TOL * max(1, z^2) * p  (relative error of a normal tail ~ z^2 eps)
DUMP_BYTES = 64_000_000  # --dump-outputs writes at most this much
DUMP_SEED = 7001


def w_smem(n):
    """Algorithmic shared-memory bytes per pair (SURVEY.md 8d): 8 * n * ceil(log2 n)."""
    return 8.0 * n * math.ceil(math.log2(max(n, 2)))


class ClockSampler:
    def __init__(self, index):
        self.rows, self.proc = [], None
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={index}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
                for k, nm in enumerate(names):
                    if r[3 + k].lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": float(np.max(mx)) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def workload_shape(name, n_gpus, scaling, cols=0, rows=0):
    from icikendalltau_b200 import synth
    n, C, q, persp, kind = synth.WORKLOADS[name]
    if cols:
        C = cols
    if rows:
        n = rows
    if scaling == "weak" and n_gpus > 1:
        # pairs ~ C^2/2: keep pairs per GPU constant
        C = int(round(math.sqrt(n_gpus * C * (C - 1) + 0.25) + 0.5))
    return n, C, persp


def workload_label(name, n, C, persp):
    """One string for both arms (the driver compares them)."""
    what = {"config1": "yeast RNA-seq counts (bundled data), zeros missing",
            "config4": "count data, heavy ties, zeros missing"}.get(name, "20-25% left-censored")
    return f"{name}: {n} features x {C} samples, {what}, {persp}"


def cpu_port_rate(x, persp, budget_s, cores):
    """Times the oracle (reference restatement) on `cores` threads on a bounded sample of pairs."""
    from oracle import oracle as O
    n, C = x.shape
    pi, pj = O.setup_comparisons(C, None, True)
    P = pi.size
    rng = np.random.default_rng(12345)
    probe = rng.choice(P, size=min(P, cores), replace=False)
    t0 = time.perf_counter()
    O.pair_loop(x, pi[probe], pj[probe], perspective=persp, ncore=cores)
    t_probe = max(time.perf_counter() - t0, 1e-4)  # ~ one pair per core
    m = int(min(P, max(cores, budget_s / t_probe * cores)))
    sel = np.sort(rng.choice(P, size=m, replace=False)) if m < P else np.arange(P)
    t0 = time.perf_counter()
    O.pair_loop(x, pi[sel], pj[sel], perspective=persp, ncore=cores)
    dt = time.perf_counter() - t0
    sample = (f"all {P} pairs" if m == P else f"seeded random sample of {m} of {P} pairs") + \
        f", {dt:.1f} s on {cores} threads, contiguous chunks of ceil(P/ncore) like furrr"
    return m / dt, sample


def run_reference(args, rank, world):
    if rank != 0:
        return
    from icikendalltau_b200 import synth
    n, C, persp = workload_shape(args.workload, args.gpus, args.scaling, args.cols, args.rows)
    x, _ = synth.make(args.workload, n=n, C=C)
    cores = os.cpu_count() or 1
    P = C * (C - 1) // 2
    rates, sample = [], ""
    for _ in range(args.warmup):
        cpu_port_rate(x, persp, 1.0, cores)
    t_all = time.perf_counter()
    for _ in range(args.steps):
        r, sample = cpu_port_rate(x, persp, args.ref_budget, cores)
        rates.append(r)
    wall = time.perf_counter() - t_all
    val = float(np.mean(rates))
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": "pairs/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * wall / max(args.steps, 1),
        "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "int64+f64",
        "data": "bundled yeast_missing" if args.workload == "config1" else "synthetic",
        "config": {"workload": workload_label(args.workload, n, C, persp), "pairs": P,
                   "note": "R/Rcpp absent from this image: reference arm = C++ restatement of "
                           "src/kendallc.cpp (oracle/), threads stand in for furrr workers; each step "
                           "times a bounded seeded sample of the workload's pairs"},
        "feature_pairs_per_sec": val * n,
        "cpu_baseline": {"value": val, "unit": "pairs/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def parity_sample(x, persp, got, lo, hi, n_sample, device):
    """Post-timing check of a seeded sample of this rank's pairs against the CPU oracle: the results
    of the TIMED plan (tau, tau_max, completeness, p-value, status) and, through a pair-list call on
    the same pairs, the integer counts (dis, ntie, xtie, ytie, tot, n_entry, b) bit-exact."""
    import icikendalltau_b200 as ik
    from oracle import oracle as O
    n, C = x.shape
    pi, pj = O.setup_comparisons(C, None, True)
    rng = np.random.default_rng(2024)
    m = min(n_sample, hi - lo)
    sel = np.sort(rng.choice(hi - lo, size=m, replace=False)) + lo
    t0 = time.perf_counter()
    ref = O.pair_loop(x, pi[sel], pj[sel], perspective=persp, ncore=os.cpu_count() or 1, want_counts=True,
                      want_z=True)
    t_ref = time.perf_counter() - t0
    lst = ik.run_pairs(x, (), pi=pi[sel], pj=pj[sel], want_counts=True, perspective=persp, device=device)
    k = sel - lo
    ok = ref["status"] == 0
    out = {"pairs": int(m), "oracle_s": round(t_ref, 2)}
    out["status_equal"] = bool(np.array_equal(got["status"][k], ref["status"]))
    out["counts_exact"] = bool(np.array_equal(lst["counts"][ok], ref["counts"][ok]))
    out["timed_equals_pair_list"] = bool(all(
        np.array_equal(got[f][k], lst[f], equal_nan=True) for f in ("raw", "pvalue", "taumax", "completeness")))

    def rel(a, b):
        a, b = a[ok], b[ok]
        with np.errstate(divide="ignore", invalid="ignore"):
            r = np.abs(a - b) / np.abs(b)
        r[(a == b)] = 0.0
        return float(np.max(r)) if r.size else 0.0

    out["tau_max_rel_err"] = rel(got["raw"][k], ref["raw"])
    out["taumax_max_rel_err"] = rel(got["taumax"][k], ref["taumax"])
    out["completeness_equal"] = bool(np.array_equal(got["completeness"][k][ok], ref["completeness"][ok]))
    pg, pr, z = got["pvalue"][k][ok], ref["pvalue"][ok], ref["z"][ok]
    with np.errstate(divide="ignore", invalid="ignore"):
        pe = np.abs(pg - pr) / (np.maximum(1.0, z * z) * np.abs(pr))
    pe[pg == pr] = 0.0
    pe[np.isnan(pg) & np.isnan(pr)] = 0.0
    out["pvalue_max_err_over_z2"] = float(np.nanmax(pe)) if pe.size else 0.0
    out["pvalue_nonzero"] = int(np.count_nonzero(pr))
    out["ok"] = bool(out["status_equal"] and out["counts_exact"] and out["timed_equals_pair_list"] and
                     out["tau_max_rel_err"] <= 1e-12 and out["taumax_max_rel_err"] <= 1e-12 and
                     out["completeness_equal"] and out["pvalue_max_err_over_z2"] <= P_TOL and
                     not np.isnan(pe).any())
    return out


def dump_outputs(out_dir, res, P):
    """Writes the per-pair results `res` (all P pairs in pair order, as Plan.download returns them) to
    out_dir/<name>.npy: raw, pvalue, taumax, completeness (float64), status (float32), max_taumax
    (float64, one element) and pair_index (float64), the positions in the pair order of the pairs
    written.  All pairs when they fit in DUMP_BYTES, otherwise a seeded random sample that depends
    only on P, so that runs of the same workload write the same pairs."""
    per_pair = 4 * 8 + 4 + 8
    m = min(P, (DUMP_BYTES - 4096) // per_pair)  # 4096: the .npy headers
    if m == P:
        sel = np.arange(P)
    else:
        sel = np.sort(np.random.default_rng(DUMP_SEED).choice(P, size=m, replace=False))
    arrays = {k: np.ascontiguousarray(res[k][sel], dtype=np.float64)
              for k in ("raw", "pvalue", "taumax", "completeness")}
    arrays["status"] = res["status"][sel].astype(np.float32)
    arrays["max_taumax"] = np.array([res["max_taumax"]], dtype=np.float64)
    arrays["pair_index"] = sel.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="target",
                    choices=["config1", "config2", "config3", "config4", "config5", "target"])
    ap.add_argument("--scaling", default="strong", choices=["weak", "strong"])
    ap.add_argument("--cpu-budget", type=float, default=15.0, help="seconds of CPU baseline (N=1 only)")
    ap.add_argument("--ref-budget", type=float, default=8.0, help="seconds per reference-arm step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--kernel", default="tiled", choices=["tiled", "naive"])
    ap.add_argument("--cols", type=int, default=0, help="override the number of samples (profiling runs only)")
    ap.add_argument("--rows", type=int, default=0, help="override the number of features (profiling runs only)")
    ap.add_argument("--quick", action="store_true", help="skip the e2e, parity and CPU legs (tuning sweeps)")
    ap.add_argument("--parity-pairs", type=int, default=320)
    ap.add_argument("--replicate-k1", action="store_true", help="N > 1: every rank preprocesses all columns")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the timed plan's results of the last step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs: the reference arm times a sample of pairs, not the whole result")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return 0
    if args.warmup < 3:
        args.warmup = 3  # timing rule: at least 3 warm-up steps

    import torch
    import torch.distributed as dist

    import icikendalltau_b200 as ik
    from icikendalltau_b200 import _lib, sharding, synth

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: libicikt_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    n_gpus = world

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v):
        if world == 1:
            return float(v)
        t = torch.tensor([float(v)], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    n, C, persp = workload_shape(args.workload, n_gpus, args.scaling, args.cols, args.rows)
    x, _ = synth.make(args.workload, n=n, C=C)  # same seed on every rank
    P_total = C * (C - 1) // 2
    lo, hi = sharding.pair_range(P_total, rank, world)
    c_lo, c_hi = sharding.column_range(C, rank, world)
    P_rank = hi - lo
    kernel = _lib.KERNEL_NAIVE if args.kernel == "naive" else _lib.KERNEL_TILED
    shard_k1 = world > 1 and not args.replicate_k1

    # pinned host copy of the matrix: the e2e leg uploads from here every step
    host = torch.empty((C, n), dtype=torch.float64, pin_memory=True)  # column-major n x C
    host.numpy()[...] = x.T
    x_pinned = host.numpy().T  # (n, C) Fortran-ordered view of the pinned buffer
    assert x_pinned.flags["F_CONTIGUOUS"]

    smem32, smem128 = _lib.measure_smem_bandwidth(local_rank)
    smem_peak = max(smem32, smem128)
    issue_alu, issue_fma, issue_mixed = _lib.measure_issue_rate(local_rank)  # G warp-instructions/s

    plan = ik.Plan(n, C, perspective=persp, device=local_rank, kernel=kernel, pair_lo=lo, pair_hi=hi)
    plan.upload(x_pinned)
    stream = torch.cuda.ExternalStream(plan.stream(), device=torch.device("cuda", local_rank))
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")  # > 126 MB L2
    gna = ()  # the synthetic matrices carry NaN for missing
    n_coll = [0]

    def step():
        if shard_k1:
            plan.columns_range(gna, c_lo, c_hi)
            n_coll[0] = sharding.exchange_tables(plan, rank, world, stream)
            plan.columns_finish()
        else:
            plan.columns(gna)
        plan.pairs()

    for _ in range(args.warmup):
        step()
    plan.sync()

    sampler = ClockSampler(local_rank)
    ev0 = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    ev1 = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    k2_ms, k1_ms, k3_ms, launches = [], [], [], 0
    barrier()
    for s in range(args.steps):
        flush.zero_()  # evict the tables from L2 between timed steps
        if world > 1:
            dist.barrier()  # strong scaling: the ranks start a step together
        torch.cuda.synchronize()
        ev0[s].record(stream)
        step()
        ev1[s].record(stream)
        plan.sync()
        t = plan.timings()
        k1_ms.append(t["columns_ms"])
        k2_ms.append(t["pairs_ms"])
        k3_ms.append(t["epilogue_ms"])
        launches += t["n_launches"]
    barrier()
    dev_ms = sum(a.elapsed_time(b) for a, b in zip(ev0, ev1))
    dev_ms = max_over_ranks(dev_ms)
    clocks = sampler.stop()
    value = P_total * args.steps / (dev_ms * 1e-3)
    # the timed plan's results of this rank's slice
    got = plan.download() if not args.quick or args.dump_outputs else None
    if args.dump_outputs:
        parts = [got]
        if world > 1:
            parts = [None] * world
            dist.all_gather_object(parts, got)
        if rank == 0:
            dump_outputs(args.dump_outputs, sharding.gather_results(parts, P_total), P_total)

    # ---- e2e: host buffers in, host results out, every step uploads and downloads ----
    e2e_kw = dict(perspective=persp, device=local_rank, kernel=kernel, pair_lo=lo, pair_hi=hi)

    def e2e_step(src):
        if world == 1:
            return ik.run_pairs(src, gna, **e2e_kw)  # the one-shot C-ABI call (icikt_all_pairs)
        if shard_k1:
            plan.upload_columns(src, c_lo, c_hi)
        else:
            plan.upload(src)
        step()
        return plan.download()

    def e2e_time(src, steps):
        for _ in range(2):
            e2e_step(src)
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            res = e2e_step(src)
        torch.cuda.synchronize()
        return max_over_ranks(time.perf_counter() - t0) / steps, res

    if args.quick:
        e2e_s, res = e2e_time(x_pinned, 1)
        e2e_pg_s = None
    else:
        e2e_s, res = e2e_time(x_pinned, args.steps)
        e2e_pg_s, _ = e2e_time(x, max(1, min(args.steps, 5)))  # plain NumPy array, fresh outputs
    h2d = n * (c_hi - c_lo if shard_k1 else C) * 8
    d2h = P_rank * (4 * 8 + 4) + 8
    api = ("icikt_all_pairs (one-shot C ABI, cached workspace)" if world == 1 else
           "plan API per rank: upload_columns + columns_range + NCCL all-gather of the tables + pairs + download")

    # ---- roofline of the dominant kernel (K2) ----
    k2_avg_ms = float(np.mean(k2_ms))
    achieved = w_smem(n) * P_rank / (k2_avg_ms * 1e-3) / 1e9
    traffic = None
    prof = os.path.join(ROOT, "profiles", "k2_dram_traffic.json")
    if os.path.exists(prof):
        try:
            traffic = json.load(open(prof)).get(args.workload)
        except Exception:
            traffic = None
    # INT/issue roofline: the pair kernel's executed warp instructions per pair come from the ncu
    # capture of the same workload (smsp__inst_executed.sum / pairs, profiles/k2_inst_per_pair.json);
    # the denominator is measured live (LOP3 and IMAD interleaved, both integer-capable pipes busy)
    issue = None
    try:
        ent = json.load(open(os.path.join(ROOT, "profiles", "k2_inst_per_pair.json"))).get(args.workload)
        if ent and args.kernel == "tiled":
            ach = ent["warp_inst_per_pair"] * P_rank / (k2_avg_ms * 1e-3) / 1e9
            issue = {"achieved": ach, "peak": issue_mixed, "unit": "G warp-inst/s", "frac": ach / issue_mixed,
                     "warp_inst_per_pair": ent["warp_inst_per_pair"], "inst_source": ent["source"],
                     "peak_source": f"measured on this GPU by icikt_measure_issue_rate: LOP3 only {issue_alu:.0f}, "
                                    f"IMAD only {issue_fma:.0f}, interleaved {issue_mixed:.0f} G warp-inst/s"}
    except Exception:
        issue = None
    hbm_peak = None
    try:
        hbm_peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]
    except Exception:
        pass

    line = {
        "metric": METRIC, "value": value, "unit": "pairs/s", "n_gpus": n_gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dev_ms / args.steps, "higher_is_better": True,
        "scaling": args.scaling, "vs_baseline": None, "dtype": "int64+f64",
        "data": "bundled yeast_missing" if args.workload == "config1" else "synthetic",
        "config": {"workload": workload_label(args.workload, n, C, persp),
                   "pairs": P_total, "pairs_per_gpu": P_rank, "kernel": args.kernel,
                   "l2": "256 MB buffer written between timed steps (L2 flushed)",
                   "parallelism": (f"pair-range x{n_gpus}; K1 sharded by columns, tables all-gathered over NCCL "
                                   f"({n_coll[0]} collectives/step); no collective on the pair path" if shard_k1 else
                                   f"pair-range x{n_gpus}, K1 replicated, no collective")},
        "feature_pairs_per_sec": value * n,
        "e2e": {"value": P_total / e2e_s, "unit": "pairs/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": 1e3 * e2e_s, "api": api + ", pinned host input"},
        "gpu_launches": launches,
        "clocks": clocks,
        "roofline": {"bound": "smem", "achieved": achieved, "peak": smem_peak, "unit": "GB/s",
                     "frac": achieved / smem_peak, "traffic": traffic,
                     "kernel": "pairs_tiled_kernel" if args.kernel == "tiled" else "pairs_naive_kernel",
                     "model": "8*n*ceil(log2 n) shared-memory bytes per pair (SURVEY.md 8d)",
                     "peak_source": f"measured on this GPU by icikt_measure_smem_bandwidth: "
                                    f"{smem32:.0f} GB/s (32-bit), {smem128:.0f} GB/s (128-bit); "
                                    "MEASURED_PEAKS.json has no shared-memory figure",
                     "issue": issue,
                     "k2_ms": k2_avg_ms, "k1_ms": float(np.mean(k1_ms)), "k3_ms": float(np.mean(k3_ms)),
                     "k2_share_of_step": k2_avg_ms * args.steps / dev_ms if world == 1 else None,
                     "k1_hbm": {"achieved_gbs": (8.0 + 4.2) * n * (c_hi - c_lo if shard_k1 else C) /
                                (np.mean(k1_ms) * 1e-3) / 1e9, "peak_gbs": hbm_peak}},
        "max_taumax": res["max_taumax"],
    }
    if world == 1 and isinstance(res.get("timings"), dict):
        # the one-shot call pipelines large jobs (column chunks uploaded behind the pair launches of earlier
        # chunks, row blocks copied out behind later ones: icikt_stage_table); its own event timings, last step
        t = res["timings"]
        line["e2e"]["launches_per_step"] = t["n_launches"]
        line["e2e"]["pipelined"] = bool(t["n_launches"] > launches // max(1, args.steps))
        line["e2e"]["device_ms"] = {k: round(float(v), 3) for k, v in t.items() if k.endswith("_ms")}
    if e2e_pg_s is not None:
        line["e2e_pageable"] = {"value": P_total / e2e_pg_s, "unit": "pairs/s", "ms_per_step": 1e3 * e2e_pg_s,
                                "api": api + ", pageable NumPy input, freshly allocated outputs"}
    if rank == 0 and not args.quick:
        line["parity_sample"] = parity_sample(x, persp, got, lo, hi, args.parity_pairs, local_rank)
    if rank == 0 and world == 1 and not args.no_cpu_baseline and not args.quick:
        cores = os.cpu_count() or 1
        rate, sample = cpu_port_rate(x, persp, args.cpu_budget, cores)
        line["cpu_baseline"] = {"value": rate, "unit": "pairs/s", "cores": cores, "kind": "port",
                                "sample": sample}
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()  # the other ranks wait for rank 0's oracle check before tearing NCCL down
    plan.close()
    _lib.release_workspace()
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
