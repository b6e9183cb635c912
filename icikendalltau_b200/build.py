"""Builds libicikt_b200.so in-tree with nvcc for sm_100a (no JIT cache, no torch extension:
the .so must travel with the repository snapshot to the GPU box)."""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libicikt_b200.so")
SOURCES = ["icikt_capi.cu", "icikt_columns.cu", "icikt_pairs.cu", "icikt_padj.cu", "icikt_reshape.cu", "icikt_select.cu"]
HEADERS = ["icikt_common.cuh", "icikt_count.cuh", "icikt_cross.cuh", "icikt_edges.cuh", "icikt_internal.h", "icikt_owned.h", "icikt_padj.cuh", "icikt_topk.cuh", os.path.join("..", "..", "include", "icikt_b200.h")]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo",
    "--fmad=false",  # keep the fp64 epilogue's operation order (no contraction)
    "-Xcompiler", "-fPIC",
]


def _nvcc() -> str:
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found; libicikt_b200.so cannot be built")
    return exe


def _stale(target: str, deps) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    nvcc = _nvcc()
    objdir = os.path.join(CSRC, "build")
    os.makedirs(objdir, exist_ok=True)
    hdrs = [os.path.join(CSRC, h) for h in HEADERS]
    objs, procs = [], []
    for src in SOURCES:
        s = os.path.join(CSRC, src)
        o = os.path.join(objdir, src.replace(".cu", ".o"))
        objs.append(o)
        if force or _stale(o, [s] + hdrs):
            cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", s, "-o", o]
            procs.append((cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)))
    for cmd, pr in procs:
        out, _ = pr.communicate()
        if verbose or pr.returncode:
            sys.stderr.write(out.decode(errors="replace"))
        if pr.returncode:
            raise RuntimeError("nvcc failed: " + " ".join(cmd))
    if force or _stale(LIB, objs):
        cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB] + objs + ["-lcudart"]
        subprocess.check_call(cmd)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
