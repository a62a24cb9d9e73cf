"""TEST INFRASTRUCTURE: host build of the render kernel's colour code (tests/hostsim/render_host.cu includes
marl_soccer_b200/csrc/render_core.cuh), so that the fp32 rasteriser can be compared with the fp64 reference on machines
without a GPU.  The product package never imports this module."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

from marl_soccer_b200 import _capi

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "hostsim", "render_host.cu")
LIB = os.path.join(HERE, "hostsim", "librender_host.so")
CSRC = os.path.join(os.path.dirname(HERE), "marl_soccer_b200", "csrc")
DEPS = (SRC, os.path.join(CSRC, "step_core.cuh"), os.path.join(CSRC, "render_core.cuh"),
        os.path.join(os.path.dirname(HERE), "include", "msoc.h"))

_lib = None


def build(force: bool = False) -> str:
    stale = (not os.path.exists(LIB)) or any(os.path.getmtime(p) > os.path.getmtime(LIB) for p in DEPS)
    if force or stale:
        subprocess.run(["nvcc", "-O2", "-std=c++17", "-Wno-deprecated-gpu-targets", "--shared", "-Xcompiler",
                        "-fPIC", "-o", LIB, SRC], check=True, capture_output=True)
    return LIB


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(LIB)
        L.rhost_render.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_void_p]
        _lib = L
    return _lib


def render(states, idx=None, height: int = 600, width: int = 800) -> np.ndarray:
    """RGB images (n, height, width, 3) uint8 of the envs `idx` (None: all) among `states` (msoc_env_state list, as
    get_states returns them): the render kernel's code on the host."""
    arr = (_capi.MsocEnvState * len(states))(*states)
    keep = None if idx is None else np.ascontiguousarray(idx, dtype=np.int64).reshape(-1)
    n = len(states) if keep is None else int(keep.size)
    out = np.empty((n, int(height), int(width), 3), np.uint8)
    lib().rhost_render(C.addressof(arr), len(states), None if keep is None else keep.ctypes.data, n, int(height),
                       int(width), out.ctypes.data)
    return out
