"""Build ``libbbd_loss.so`` in-tree with nvcc for sm_100a.

    python -m baseboostdepth_b200.build [--force]

The shared object lands next to this file (git-ignored, but it travels to the
GPU box with the working tree).  nvcc cross-compiles without a GPU.
"""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "csrc", "bbd_kernels.cu")
OUT = os.path.join(HERE, "libbbd_loss.so")
DEPS = [os.path.join(HERE, "csrc", f) for f in
        ("bbd_kernels.cu", "bbd_common.cuh", "bbd_strip.cuh", "bbd_stream.cuh", "bbd_pipe.cuh", "bbd_smooth.cuh", "bbd_ops.cuh",
         "bbd_framegrad.cuh", "bbd_launch.cuh")] + [
    os.path.join(os.path.dirname(HERE), "include", "bbd_loss.h")]

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-shared", "-Xcompiler", "-fPIC", "--fmad=true"]


def stale() -> bool:
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    return any(os.path.getmtime(d) > t for d in DEPS)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not stale():
        return OUT
    nvcc = os.environ.get("NVCC", "nvcc")
    extra = os.environ.get("BBD_NVCC_EXTRA", "").split()
    out = os.environ.get("BBD_LIB_OUT", OUT)
    cmd = [nvcc] + NVCC_FLAGS + extra + (["-Xptxas", "-v"] if verbose else []) + ["-o", out, SRC]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + res.stdout + res.stderr)
    if verbose:
        print(res.stderr)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
