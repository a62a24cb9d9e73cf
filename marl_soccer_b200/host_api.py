"""HostBufferSim -- the C-ABI of include/msoc.h driven with NumPy HOST buffers.

This is the path the NumPy drop-in classes use (soccer_env.SoccerEnv, marl_vecenv.SyncMultiAgentVecEnv):
actions are copied host->device, the fused kernel runs, observations / rewards / flags are copied back
(msoc_step_host).  The simulation itself always runs on the GPU; there is no CPU path.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _capi


class HostBufferSim:
    """pinned=True keeps ONE set of page-locked host buffers for the lifetime of the sim (allocated through torch) and
    returns views of them: the copies then run at PCIe speed instead of through the driver's bounce buffers (what bench.py
    measures as `e2e`), but the arrays a step returns are overwritten by the next step -- copy what you keep.  The default
    (fresh pageable arrays every call) has the reference's value semantics."""

    def __init__(self, n: int, config: dict, seed: int = 0, global_offset: int = 0, device: int = 0, pinned: bool = False):
        self._L = _capi.lib()
        self.n = int(n)
        self._pin = {}
        self._pinned = bool(pinned)
        self.config = config
        self._cfg = _capi.make_config(config)
        h = C.c_void_p()
        _capi.check(self._L.msoc_create(C.byref(self._cfg), self.n, int(device), int(seed) & (2**64 - 1),
                                        int(global_offset), C.byref(h)))
        self._h = h
        self.score = np.zeros((self.n, 2), np.int32)

    def close(self) -> None:
        if getattr(self, "_h", None):
            self._L.msoc_destroy(self._h)
            self._h = None

    __del__ = close

    def _out(self, name: str, shape, dtype) -> np.ndarray:
        """Output array: fresh and pageable, or the sim's persistent page-locked one."""
        if not self._pinned:
            return np.zeros(shape, dtype)
        if name not in self._pin:
            import torch
            t = torch.zeros(shape, dtype=getattr(torch, np.dtype(dtype).name), pin_memory=True)
            self._pin[name] = (t, t.numpy())  # the tensor owns the page-locked allocation
        return self._pin[name][1]

    def _in(self, actions) -> np.ndarray:
        a = np.ascontiguousarray(actions, dtype=np.float32).reshape(self.n, 12)
        if self._pinned:
            buf = self._out("actions", (self.n, 12), np.float32)
            np.copyto(buf, a)
            return buf
        return a

    def reset(self, mode: int = _capi.MODE_RANDOM, seed: int | None = None, mask=None) -> np.ndarray:
        obs = self._out("obs", (self.n, 4, 66), np.float32)
        m = None if mask is None else np.ascontiguousarray(mask, dtype=np.uint8)
        _capi.check(self._L.msoc_reset_host(self._h, None if m is None else m.ctypes.data, int(mode),
                                            0 if seed is None else 1,
                                            0 if seed is None else int(seed) & (2**64 - 1), obs.ctypes.data, None))
        return obs

    def step(self, actions, auto_reset: bool = True):
        a = self._in(actions)
        obs = self._out("obs", (self.n, 4, 66), np.float32)
        rew = self._out("rew", (self.n, 2), np.float32)
        done = self._out("done", (self.n,), np.uint8)
        goal = self._out("goal", (self.n,), np.int8)
        self.score = self._out("score", (self.n, 2), np.int32)
        _capi.check(self._L.msoc_step_host(self._h, a.ctypes.data, obs.ctypes.data, rew.ctypes.data,
                                           done.ctypes.data, goal.ctypes.data, self.score.ctypes.data,
                                           _capi.STEP_AUTO_RESET if auto_reset else 0, None))
        return obs, rew, done, goal

    def step_frames(self, actions, auto_reset: bool = True):
        """msoc_step_host_frames: like step(), but only the newest 22-float frame of every agent comes back, (N,4,22) --
        a third of the D2H bytes.  The caller owns the 3-frame stack: append the frame; where `done` is set (and
        auto_reset) the frame is the first one of the next episode and fills all three slots."""
        a = self._in(actions)
        frames = self._out("frames", (self.n, 4, 22), np.float32)
        rew = self._out("rew", (self.n, 2), np.float32)
        done = self._out("done", (self.n,), np.uint8)
        goal = self._out("goal", (self.n,), np.int8)
        self.score = self._out("score", (self.n, 2), np.int32)
        _capi.check(self._L.msoc_step_host_frames(self._h, a.ctypes.data, frames.ctypes.data, rew.ctypes.data,
                                                  done.ctypes.data, goal.ctypes.data, self.score.ctypes.data,
                                                  _capi.STEP_AUTO_RESET if auto_reset else 0, None))
        return frames, rew, done, goal

    def get_states(self, idx) -> list:
        idx = np.ascontiguousarray(idx, dtype=np.int64)
        arr = (_capi.MsocEnvState * len(idx))()
        _capi.check(self._L.msoc_get_state(self._h, idx.ctypes.data, len(idx), C.byref(arr)))
        return list(arr)

    def set_states(self, idx, states) -> None:
        """Injects states.  The observation history travels inside the state (hist_* poses, include/msoc.h):
        with hist_valid = 0 the frames already emitted stay what they were."""
        idx = np.ascontiguousarray(idx, dtype=np.int64)
        arr = (_capi.MsocEnvState * len(idx))(*states)
        _capi.check(self._L.msoc_set_state(self._h, idx.ctypes.data, len(idx), C.byref(arr)))

    def save_states(self, idx) -> np.ndarray:
        """States of the envs idx as an array of _capi.ENV_STATE_DTYPE (msoc_get_state straight into it).  The bytes are
        the device format of BatchedSoccerSim.save_states:
        torch.from_numpy(arr.view(np.uint8).reshape(n, 808)) moves a snapshot to the device."""
        idx = np.ascontiguousarray(idx, dtype=np.int64).reshape(-1)
        arr = np.zeros(idx.size, _capi.ENV_STATE_DTYPE)
        if idx.size:
            _capi.check(self._L.msoc_get_state(self._h, idx.ctypes.data, idx.size, arr.ctypes.data))
        return arr

    def load_states(self, idx, arr) -> None:
        """Installs an array of _capi.ENV_STATE_DTYPE (or (n, 808) uint8) into the envs idx (msoc_set_state)."""
        idx = np.ascontiguousarray(idx, dtype=np.int64).reshape(-1)
        arr = np.ascontiguousarray(arr)
        if arr.dtype != _capi.ENV_STATE_DTYPE:
            arr = arr.view(np.uint8).reshape(-1).view(_capi.ENV_STATE_DTYPE)
        if arr.size != idx.size:
            raise ValueError(f"{idx.size} indices for {arr.size} states")
        if idx.size:
            _capi.check(self._L.msoc_set_state(self._h, idx.ctypes.data, idx.size, arr.ctypes.data))

    def get_state(self, i: int):
        return self.get_states([i])[0]

    def set_state(self, i: int, S) -> None:
        self.set_states([i], [S])

    def get_obs(self, i: int) -> np.ndarray:
        idx = np.array([i], np.int64)
        o = np.zeros((1, 4, 66), np.float32)
        _capi.check(self._L.msoc_get_obs_host(self._h, idx.ctypes.data, 1, o.ctypes.data))
        return o[0]

    def render(self, idx=None, height: int = 600, width: int = 800) -> np.ndarray:
        """RGB images (n, height, width, 3) uint8 of the envs `idx` (None: all), drawn on the device and copied back
        (msoc_render_host); an index out of range raises."""
        if idx is None:
            n, iptr, keep = self.n, None, None
        else:
            keep = np.ascontiguousarray(idx, dtype=np.int64).reshape(-1)
            n, iptr = int(keep.size), keep.ctypes.data
        out = np.empty((n, int(height), int(width), 3), np.uint8)
        _capi.check(self._L.msoc_render_host(self._h, iptr, n, int(height), int(width), out.ctypes.data))
        return out

    def counters(self):
        score = np.zeros((self.n, 2), np.int32)
        steps = np.zeros((self.n,), np.int32)
        _capi.check(self._L.msoc_read_counters(self._h, score.ctypes.data, steps.ctypes.data, None))
        return score, steps

    def stats(self, reset: bool = False) -> dict:
        s = _capi.MsocStats()
        _capi.check(self._L.msoc_stats_read(self._h, C.byref(s), 1 if reset else 0, None))
        return {k: getattr(s, k) for k, _ in _capi.MsocStats._fields_}
