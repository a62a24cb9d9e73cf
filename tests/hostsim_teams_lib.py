"""TEST INFRASTRUCTURE: the host harness with red's reward (tests/hostsim/hostsim_teams.cu = hostsim.cu plus
hsim_step_teams, the host build of msoc_step_teams).  TeamsHostSim is hostsim_lib.HostSim on that library;
step(team_rewards=True) returns the (n, 4) reward with red's in columns 2, 3."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

import hostsim_lib
from marl_soccer_b200 import _capi

SRC = os.path.join(hostsim_lib.HERE, "hostsim", "hostsim_teams.cu")
LIB = os.path.join(hostsim_lib.HERE, "hostsim", "libhostsim_teams.so")

_lib = None


def build(force: bool = False) -> str:
    stale = (not os.path.exists(LIB)) or any(
        os.path.getmtime(p) > os.path.getmtime(LIB) for p in (SRC, hostsim_lib.SRC, hostsim_lib.CORE))
    if force or stale:
        subprocess.run(["nvcc", "-O2", "-std=c++17", "-Wno-deprecated-gpu-targets", "--shared", "-Xcompiler",
                        "-fPIC", "-o", LIB, SRC], check=True, capture_output=True)
    return LIB


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(LIB)
        vp, u64, i64 = C.c_void_p, C.c_uint64, C.c_int64
        L.hsim_create.restype = vp
        L.hsim_create.argtypes = [C.POINTER(_capi.MsocConfig), i64, u64, u64, vp]
        L.hsim_destroy.argtypes = [vp]
        L.hsim_reset.argtypes = [vp, vp, C.c_int, C.c_int, u64, vp]
        L.hsim_step.argtypes = [vp, vp, vp, vp, vp, vp, vp, C.c_uint32]
        L.hsim_step_teams.argtypes = [vp, vp, vp, vp, vp, vp, vp, C.c_uint32]
        L.hsim_stats.argtypes = [vp, vp, C.c_int]
        L.hsim_last.argtypes = [vp, vp, vp]
        L.hsim_get_state.argtypes = [vp, i64, C.POINTER(_capi.MsocEnvState)]
        L.hsim_set_state.argtypes = [vp, i64, C.POINTER(_capi.MsocEnvState)]
        _lib = L
    return _lib


class TeamsHostSim(hostsim_lib.HostSim):
    name = "hostsim_teams"

    def __init__(self, n: int, config: dict, seed: int = 0, global_offset: int = 0):
        self._L = lib()
        self.n = int(n)
        self._cfg = _capi.make_config(config)
        self.obs = np.zeros((self.n, 4, 66), np.float32)
        self._h = self._L.hsim_create(C.byref(self._cfg), self.n, seed, global_offset, self.obs.ctypes.data)

    def step(self, actions, auto_reset: bool = True, team_rewards: bool = False):
        """team_rewards: the step of msoc_step_teams, reward (n, 4) with red's in columns 2, 3; otherwise hsim_step."""
        if not team_rewards:
            return super().step(actions, auto_reset)
        a = np.ascontiguousarray(actions, dtype=np.float32).reshape(self.n, 12)
        out = np.zeros_like(self.obs)
        rew = np.zeros((self.n, 4), np.float32)
        done = np.zeros(self.n, np.uint8)
        goal = np.zeros(self.n, np.int8)
        self.score = np.zeros((self.n, 2), np.int32)
        self._L.hsim_step_teams(self._h, a.ctypes.data, out.ctypes.data, rew.ctypes.data,
                                done.ctypes.data, goal.ctypes.data, self.score.ctypes.data, 1 if auto_reset else 0)
        self.obs = out
        return out.copy(), rew, done, goal
