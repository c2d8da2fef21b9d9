"""Build liblogreg_b200.so in-tree with nvcc for sm_100a (B200).

    python -m logreg_b200.build [--force]

nvcc cross-compiles without a GPU; the .so is git-ignored but travels to the GPU
box with the gpurun snapshot.
"""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG)
CSRC = os.path.join(PKG, "csrc")
LIBDIR = os.path.join(PKG, "_lib")
LIB = os.path.join(LIBDIR, "liblogreg_b200.so")
STAMP = os.path.join(LIBDIR, "liblogreg_b200.srchash")

SOURCES = ["lrb_api.cu"]
HEADERS = ["common.cuh", "sampler.cuh", "eval_kernel.cuh", "eval_mc_kernel.cuh", "eval_tc_kernel.cuh", "eval_persist_kernel.cuh", "newton.cuh", "data.cuh", "predictive.cuh", "loo.cuh"]


def nccl_include() -> str:
    try:
        import nvidia.nccl as m  # bundled with torch
        inc = os.path.join(list(m.__path__)[0], "include")
        if os.path.exists(os.path.join(inc, "nccl.h")):
            return inc
    except Exception:
        pass
    return "/usr/include"


def nccl_library() -> str:
    """Path of the libnccl.so.2 the library should dlopen (torch's bundled copy first)."""
    try:
        import nvidia.nccl as m
        cand = os.path.join(list(m.__path__)[0], "lib", "libnccl.so.2")
        if os.path.exists(cand):
            return cand
    except Exception:
        pass
    return "libnccl.so.2"


def source_hash() -> str:
    h = hashlib.sha256()
    files = [os.path.join(CSRC, f) for f in SOURCES + HEADERS] + [os.path.join(ROOT, "include", "logreg_b200.h")]
    for f in files:
        with open(f, "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()


def nvcc_path() -> str:
    for c in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if c and os.path.exists(c):
            return c
    raise RuntimeError("nvcc not found: cannot build liblogreg_b200.so")


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(LIBDIR, exist_ok=True)
    want = source_hash()
    if not force and os.path.exists(LIB) and os.path.exists(STAMP) and open(STAMP).read().strip() == want:
        return LIB
    cmd = [nvcc_path(),
           "-gencode", "arch=compute_100a,code=sm_100a",
           "-O3", "-lineinfo", "-std=c++17",
           "-fmad=false",  # contraction only where the kernels ask for it (explicit fma): keeps the
                           # sampler arithmetic in the reference's (NumPy, unfused) rounding
           "-Xcompiler", "-fPIC", "-shared",
           "-I", nccl_include(),
           *[os.path.join(CSRC, s) for s in SOURCES],
           "-o", LIB, "-ldl"]
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
        print(" ".join(cmd), flush=True)
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + r.stdout + r.stderr)
    if verbose:
        print(r.stderr)
    with open(STAMP, "w") as fh:
        fh.write(want)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
