"""In-tree build of libaerobulk_gpu.so for sm_100a (nvcc cross-compiles without a GPU).

    python -m aerobulk_b200.build [--force]

The shared library lands next to this file (git-ignored, shipped to the GPU box by
gpurun).  No JIT cache, no torch extension machinery: six translation units,
one link step.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
ROOT = os.path.dirname(HERE)
LIB = os.path.join(HERE, "libaerobulk_gpu.so")
OBJ = os.path.join(HERE, "build")

ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
NVCC_FLAGS = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden"]
# -fmad=true (default): FMA contraction is part of the documented GPU arithmetic (DESIGN.md)

SOURCES = ["ab_kernels.cu", "ab_series.cu", "ab_ice.cu", "ab_probe.cu", "ab_api.cu", "aerobulk.cpp"]
HEADERS = [os.path.join(CSRC, h) for h in ("ab_device.cuh", "ab_ice.cuh", "ab_kernels.cuh", "ab_math.cuh", "ab_math_tables.cuh", "ab_copy_pool.hpp")] + [
    os.path.join(ROOT, "include", h) for h in ("aerobulk_gpu.h", "aerobulk.hpp")]


def _nvcc() -> str:
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found: cannot build libaerobulk_gpu.so")
    return exe


def _stale(target: str, deps) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    """Build the library."""
    os.makedirs(OBJ, exist_ok=True)
    nvcc = _nvcc()
    objs = []
    jobs = []
    for src in SOURCES:
        path = os.path.join(CSRC, src)
        obj = os.path.join(OBJ, os.path.splitext(src)[0] + ".o")
        objs.append(obj)
        if force or _stale(obj, [path] + HEADERS):
            cmd = [nvcc, "-ccbin", "/usr/bin/g++"] + ARCH + NVCC_FLAGS + ["-c", path, "-o", obj]
            if src.endswith(".cu") and verbose:
                cmd += ["-Xptxas", "-v"]
            if verbose:
                print(" ".join(cmd), flush=True)
            jobs.append((cmd, subprocess.Popen(cmd)))   # the translation units compile side by side
    for cmd, job in jobs:
        if job.wait() != 0:
            raise subprocess.CalledProcessError(job.returncode, cmd)
    if force or _stale(LIB, objs):
        # -z nodelete: the copy threads of ab_copy_pool.hpp must outlive any dlclose of the library
        cmd = [nvcc, "-ccbin", "/usr/bin/g++"] + ARCH + ["-shared", "-o", LIB] + objs + [
            "-cudart", "static", "-Xlinker", "--exclude-libs,ALL", "-Xlinker", "-z", "-Xlinker", "nodelete"]
        if verbose:
            print(" ".join(cmd), flush=True)
        subprocess.check_call(cmd)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
