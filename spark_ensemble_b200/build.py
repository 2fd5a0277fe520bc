"""Builds libse_b200.so (the C-ABI of include/se_abi.h) for sm_100a with nvcc, in-tree.

    python -m spark_ensemble_b200.build [--force]

The shared library lands in spark_ensemble_b200/lib/ (git-ignored, travels to the GPU box).
"""
from __future__ import annotations

import concurrent.futures as cf
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
OBJDIR = os.path.join(LIBDIR, "obj")
LIB = os.path.join(LIBDIR, "libse_b200.so")
SOURCES = ["se_api.cu", "se_gbm.cu", "se_gbm_tiled.cu", "se_gbm_fused.cu", "se_gbm_generic.cu", "se_brent.cu", "se_boost.cu", "se_agg.cu", "se_models.cu", "se_util.cu"]
# the device Brent must round every multiply and add separately to reproduce the host line search bit for bit
EXTRA_FLAGS = {"se_brent.cu": ["-fmad=false"], "se_gbm_fused.cu": ["-fmad=false"]}
HEADERS = ["se_common.cuh", "se_kernels.h", "se_loss.cuh", "se_tma.cuh", "se_brent.h", "se_sortnet.h", "se_wmedian.cuh", os.path.join("..", "..", "include", "se_abi.h")]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def _stale(target: str, deps: list[str]) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(OBJDIR, exist_ok=True)
    nvcc = _nvcc()
    hdrs = [os.path.join(CSRC, h) for h in HEADERS]
    jobs = []
    for src in SOURCES:
        s = os.path.join(CSRC, src)
        o = os.path.join(OBJDIR, src.replace(".cu", ".o"))
        if force or _stale(o, [s] + hdrs):
            jobs.append((s, o))

    def compile_one(job):
        s, o = job
        cmd = [nvcc] + NVCC_FLAGS + EXTRA_FLAGS.get(os.path.basename(s), []) + ["-c", s, "-o", o]
        if verbose:
            print(" ".join(cmd), flush=True)
        subprocess.check_call(cmd)

    if jobs:
        with cf.ThreadPoolExecutor(max_workers=min(len(jobs), os.cpu_count() or 4)) as ex:
            list(ex.map(compile_one, jobs))
    objs = [os.path.join(OBJDIR, s.replace(".cu", ".o")) for s in SOURCES]
    if jobs or force or _stale(LIB, objs):
        cmd = [nvcc, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a",
                                                    "-Xcompiler", "-fPIC", "-ldl"]
        if verbose:
            print(" ".join(cmd), flush=True)
        subprocess.check_call(cmd)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
