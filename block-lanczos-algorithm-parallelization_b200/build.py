"""Build recipes: the CUDA shared library (sm_100a) and the C host driver.

Everything is built IN-TREE so that the artefacts travel to the GPU box with the repo
snapshot.  nvcc cross-compiles without a GPU.
"""
from __future__ import annotations

import glob
import os
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG)
CSRC = os.path.join(PKG, "csrc")
LIB = os.path.join(PKG, "libblklanczos.so")
DRIVER_DIR = os.path.join(PKG, "driver")
DRIVER = os.path.join(DRIVER_DIR, "lanczos_modp")

NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
CU_SOURCES = ["layout_build.cu", "spmv.cu", "dense.cu", "dense_mma.cu", "dense_umma.cu", "loop_coop.cu", "kernel_basis.cu", "solve.cu", "prune.cu", "context.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-Wall", "-ccbin", "/usr/bin/g++"]


def _stale(target: str, sources: list[str]) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(s) > t for s in sources)


def build_library(force: bool = False, verbose: bool = False) -> str:
    srcs = [os.path.join(CSRC, s) for s in CU_SOURCES]
    # every header any translation unit can include: editing one of them must rebuild the library
    deps = srcs + sorted(glob.glob(os.path.join(CSRC, "*.cuh"))) + sorted(glob.glob(os.path.join(ROOT, "include", "*.h")))
    if not force and not _stale(LIB, deps):
        return LIB
    objs = []
    procs = []
    for s in srcs:
        o = s[:-3] + ".o"
        objs.append(o)
        cmd = [NVCC, *NVCC_FLAGS, "-c", s, "-o", o] + (["-Xptxas", "-v"] if verbose else [])
        procs.append((cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for cmd, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode:
            sys.stderr.write(out)
        if p.returncode:
            raise RuntimeError("nvcc failed: " + " ".join(cmd))
    subprocess.check_call([NVCC, "-shared", "-o", LIB, *objs, "-ccbin", "/usr/bin/g++", "-ldl"])
    return LIB


def build_driver(force: bool = False) -> str:
    srcs = [os.path.join(DRIVER_DIR, f) for f in ("lanczos_modp_gpu.c", "mtx_io.c")]
    if not all(os.path.exists(s) for s in srcs):
        raise FileNotFoundError("driver sources missing")
    build_library()
    if force or _stale(DRIVER, srcs + [LIB, os.path.join(DRIVER_DIR, "mtx_io.h")]):
        subprocess.check_call(["/usr/bin/gcc", "-std=c99", "-O2", "-Wall", "-Wextra", "-Werror",
                               "-I", os.path.join(ROOT, "include"), *srcs, "-o", DRIVER,
                               "-L", PKG, "-lblklanczos", "-Wl,-rpath,$ORIGIN/..", "-lm", "-lpthread"])
    return DRIVER


if __name__ == "__main__":
    build_library(force="--force" in sys.argv, verbose="-v" in sys.argv)
    if os.path.exists(os.path.join(DRIVER_DIR, "lanczos_modp_gpu.c")):
        build_driver(force="--force" in sys.argv)
    print(LIB)
