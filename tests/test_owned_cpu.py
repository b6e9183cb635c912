"""The owning handles of the host code (icikendalltau_b200/csrc/icikt_owned.h) without a GPU: tests/owned_host.cpp,
built with g++ against the CUDA runtime with its memory calls wrapped by a fake allocator, checks that reserve keeps or
replaces an allocation, that a failed reserve leaves an empty handle and the next one tries again, and that moves
transfer ownership so that every allocation is freed exactly once."""
import os
import subprocess

from icikendalltau_b200 import build

HERE = os.path.dirname(os.path.abspath(__file__))


def test_owned_handles(tmp_path):
    cuda = os.path.dirname(os.path.dirname(os.path.realpath(build._nvcc())))
    lib = os.path.join(cuda, "lib64")
    exe = str(tmp_path / "owned_host")
    wrap = ",".join("--wrap=" + f for f in ("cudaMalloc", "cudaMallocHost", "cudaFree", "cudaFreeHost"))
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-I", os.path.join(cuda, "include"),
                           os.path.join(HERE, "owned_host.cpp"), "-o", exe, "-L", lib, "-Wl,-rpath," + lib,
                           "-Wl," + wrap, "-lcudart"])
    r = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and r.stdout.strip().endswith("ok"), r.stdout + r.stderr
