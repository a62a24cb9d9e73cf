"""Builds marl_soccer_b200/libmsoc.so (hand-written sm_100a kernels + C-ABI) in-tree with nvcc.

    python -m marl_soccer_b200.build [--force]
"""
from __future__ import annotations

import os
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG)
SRC = os.path.join(PKG, "csrc", "msoc.cu")
DEPS = [SRC, os.path.join(PKG, "csrc", "step_core.cuh"), os.path.join(PKG, "csrc", "render_core.cuh"),
        os.path.join(ROOT, "include", "msoc.h")]
OUT = os.path.join(PKG, "libmsoc.so")
OUT_CHECKED = os.path.join(PKG, "libmsoc_checked.so")  # same sources with -DMSOC_CHECKS: the kernels' own bounds checks

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "--shared", "-Xcompiler", "-fPIC"]


def build(force: bool = False, verbose: bool = False) -> str:
    stale = (not os.path.exists(OUT)) or any(os.path.getmtime(d) > os.path.getmtime(OUT) for d in DEPS)
    if force or stale:
        nvcc = os.environ.get("NVCC", "nvcc")
        cmd = [nvcc, *NVCC_FLAGS, "-Xptxas", "-v", "-o", OUT, SRC]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if verbose or r.returncode != 0:
            sys.stderr.write(r.stdout + r.stderr)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed building libmsoc.so")
    return OUT


def build_checked(force: bool = False) -> str:
    """The debug build (tests/test_gpu_checked.py): every index the kernels compute is checked on the device."""
    stale = (not os.path.exists(OUT_CHECKED)) or any(os.path.getmtime(d) > os.path.getmtime(OUT_CHECKED) for d in DEPS)
    if force or stale:
        nvcc = os.environ.get("NVCC", "nvcc")
        r = subprocess.run([nvcc, *NVCC_FLAGS, "-DMSOC_CHECKS", "-o", OUT_CHECKED, SRC], capture_output=True, text=True)
        if r.returncode != 0:
            sys.stderr.write(r.stdout + r.stderr)
            raise RuntimeError("nvcc failed building libmsoc_checked.so")
    return OUT_CHECKED


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
    print(build_checked(force="--force" in sys.argv))
