"""BatchedSoccerSim -- the device-resident form of the reference's env stack.

N independent 2v2 soccer envs live in HBM buffers (contiguous per-env records) owned by one C-ABI handle
(include/msoc.h); one fused CUDA kernel per `step` replaces
SyncMultiAgentVecEnv.step -> SoccerEnv.step -> Game.step -> pymunk Space.step
(soccer_simulation/marl_vecenv.py:30-68, soccer_env.py:100-154, game/game.py:378-437).
Actions, observations, rewards, dones and goal flags are torch CUDA tensors; nothing crosses PCIe.

There is no CPU path: constructing a sim without the built extension or without a CUDA device raises.
"""
from __future__ import annotations

import ctypes as C
import json
import os

import numpy as np
import torch

from . import _capi

_DEFAULT_CONFIG_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "config.json")


def load_default_config() -> dict:
    """The shipped config.json (same keys and values as soccer_simulation/config.json)."""
    with open(_DEFAULT_CONFIG_PATH) as f:
        return json.load(f)


class _DevMem:
    def __init__(self, ptr, shape, typestr):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (int(ptr), False),
                                         "version": 2, "strides": None}


def _view(ptr, shape, typestr, device) -> torch.Tensor:
    with torch.cuda.device(device):
        return torch.as_tensor(_DevMem(ptr, shape, typestr), device=device)


class BatchedSoccerSim:
    """N envs on one GPU.

    step() returns views of internal buffers that stay valid until the next step():
      obs    (N, 4, 66) float32   3 stacked 22-float frames per agent, newest last (soccer_env.py:37-39)
      reward (N, 2)     float32   blue agents only; red is always 0.0 (soccer_env.py:141-146)
                (N, 4)     float32   with step(..., team_rewards=True): blue's in columns 0, 1, red's own reward in 2, 3
      done   (N,)       uint8     truncation at max_steps (soccer_env.py:148); never "terminated"
      goal   (N,)       int8      +1 blue scored, -1 red scored (info["goal_scored_by"])
      score  (N, 2)     int32     info["score"] of the step, before any auto-reset
    """

    def __init__(self, num_envs: int, config: dict | None = None, device: str | int | torch.device = "cuda:0",
                 seed: int = 0, global_env_offset: int = 0):
        if not torch.cuda.is_available():
            raise _capi.MsocError("BatchedSoccerSim needs a CUDA device (there is no CPU fallback)")
        self._L = _capi.lib()
        self.device = torch.device(device if not isinstance(device, int) else f"cuda:{device}")
        if self.device.type != "cuda":
            raise _capi.MsocError("BatchedSoccerSim runs on CUDA devices only")
        self.num_envs = int(num_envs)
        self.config = config if config is not None else load_default_config()
        self.global_env_offset = int(global_env_offset)
        self._cfg = _capi.make_config(self.config)
        dev_index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        h = C.c_void_p()
        _capi.check(self._L.msoc_create(C.byref(self._cfg), self.num_envs, dev_index, int(seed) & (2**64 - 1),
                                        self.global_env_offset, C.byref(h)))
        self._h = h
        n, d = self.num_envs, self.device
        # zero-copy torch views of the handle's device buffers (valid while the handle lives); they
        # already hold the first spawn's observation (Game.__init__ -> reset, game/game.py:43,74)
        bufs = _capi.MsocBuffers()
        _capi.check(self._L.msoc_device_buffers(self._h, C.byref(bufs)))
        self.obs = _view(bufs.obs, (n, 4, 66), "<f4", d)
        self.actions = _view(bufs.actions, (n, 4, 3), "<f4", d)
        self.reward = _view(bufs.reward, (n, 2), "<f4", d)
        self.done = _view(bufs.done, (n,), "|u1", d)
        self.goal = _view(bufs.goal, (n,), "|i1", d)
        self.score = _view(bufs.score, (n, 2), "<i4", d)
        self._stats = torch.zeros((8,), dtype=torch.float64, device=d)
        self._stats_live = _view(bufs.stats, (8,), "<f8", d)  # the accumulators themselves (state_dict)
        self.reward4 = None  # (N, 4) rewards of step(team_rewards=True), allocated by its first call

    def _index(self, idx, unique: bool = False, n_all: int | None = None):
        """(int64 CUDA tensor or None, count) of an env index argument: None (envs 0..n_all-1, default all), a host
        sequence / ndarray / CPU tensor (checked: ValueError when out of range, or repeated with `unique`), or an int64
        CUDA tensor on the sim's device (not checked)."""
        if idx is None:
            return None, self.num_envs if n_all is None else int(n_all)
        if isinstance(idx, torch.Tensor) and idx.is_cuda:
            if idx.dtype != torch.int64 or idx.device != self.device or idx.dim() != 1:
                raise ValueError("a CUDA index tensor must be 1-D int64 on the sim's device")
            idx = idx.contiguous()
            return idx, int(idx.numel())
        host = np.asarray(idx.cpu() if isinstance(idx, torch.Tensor) else idx)
        if host.ndim != 1 or (host.size and not np.issubdtype(host.dtype, np.integer)):
            raise ValueError("idx must be a 1-D sequence of integer env indices")
        host = host.astype(np.int64)
        if host.size and (host.min() < 0 or host.max() >= self.num_envs):
            raise ValueError(f"env index out of range [0, {self.num_envs})")
        if unique and np.unique(host).size != host.size:
            raise ValueError("env indices to write must not repeat")
        return torch.from_numpy(host).to(self.device), int(host.size)

    def close(self) -> None:
        if getattr(self, "_h", None):
            self._L.msoc_destroy(self._h)
            self._h = None

    __del__ = close

    def _stream(self) -> int:
        return torch.cuda.current_stream(self.device).cuda_stream

    def reset(self, mode: int = _capi.MODE_RANDOM, seed: int | None = None, mask: torch.Tensor | None = None) -> torch.Tensor:
        """Game.reset for all (or the masked) envs; env i is seeded with seed + global index
        (marl_vecenv.py:23).  Returns the stacked observation (3 copies of frame 0, soccer_env.py:92-96)."""
        mptr = None
        if mask is not None:
            mask = mask.to(device=self.device, dtype=torch.uint8).contiguous()
            mptr = mask.data_ptr()
        _capi.check(self._L.msoc_reset(self._h, mptr, int(mode), 0 if seed is None else 1,
                                       0 if seed is None else int(seed) & (2**64 - 1), self.obs.data_ptr(),
                                       self._stream()))
        return self.obs

    def step(self, actions: torch.Tensor, auto_reset: bool = True, general_path: bool = False, team_rewards: bool = False):
        """One env-step for every env.  actions: (N, 4, 3) float32 CUDA tensor in [-1, 1] (clipped on
        the device like soccer_env.py:119).  general_path (debugging / tests): every env that touches something is
        stepped by the general contact path instead of its work class's own.
        team_rewards: step with msoc_step_teams; the reward returned is then `self.reward4` (N, 4): blue's reward
        in columns 0, 1 (what the plain step returns), red's own reward in 2, 3 (include/msoc.h).  That tensor is
        allocated by the first such call, which therefore must not be inside a CUDA graph capture."""
        if actions.device != self.device or actions.dtype != torch.float32 or not actions.is_contiguous():
            actions = actions.to(device=self.device, dtype=torch.float32).contiguous()
        if actions.numel() != self.num_envs * 12:
            raise ValueError(f"actions must have shape ({self.num_envs}, 4, 3), got {tuple(actions.shape)}")
        flags = (_capi.STEP_AUTO_RESET if auto_reset else 0) | (_capi.STEP_GENERAL_PATH if general_path else 0)
        if team_rewards:
            if self.reward4 is None:
                if torch.cuda.is_current_stream_capturing():
                    raise RuntimeError("the first step(team_rewards=True) allocates the (N, 4) reward tensor: "
                                       "call it once before capturing a CUDA graph")
                self.reward4 = torch.zeros((self.num_envs, 4), dtype=torch.float32, device=self.device)
            _capi.check(self._L.msoc_step_teams(self._h, actions.data_ptr(), self.obs.data_ptr(),
                                                self.reward4.data_ptr(), self.done.data_ptr(), self.goal.data_ptr(),
                                                self.score.data_ptr(), flags, self._stream()))
            return self.obs, self.reward4, self.done, self.goal
        _capi.check(self._L.msoc_step(self._h, actions.data_ptr(), self.obs.data_ptr(),
                                      self.reward.data_ptr(), self.done.data_ptr(), self.goal.data_ptr(),
                                      self.score.data_ptr(), flags, self._stream()))
        return self.obs, self.reward, self.done, self.goal

    def stats_tensor(self, reset: bool = False) -> torch.Tensor:
        """8 float64 on the device (msoc_stats layout): episodes, return sum, goals blue/red, env-steps,
        contacts, contact overflow -- ready for one all-reduce per rollout."""
        _capi.check(self._L.msoc_stats_device(self._h, self._stats.data_ptr(), 1 if reset else 0, self._stream()))
        return self._stats

    def stats(self, reset: bool = False) -> dict:
        t = self.stats_tensor(reset).cpu().tolist()
        return dict(zip([k for k, _ in _capi.MsocStats._fields_], t))

    def class_counts(self) -> dict:
        """Work classes of the last step (instrumentation): envs handed to the contact kernel per class."""
        out = (C.c_int32 * 4)()
        _capi.check(self._L.msoc_last_class_counts(self._h, C.byref(out), self._stream()))
        return {"light": out[0], "heavy": out[1], "pair": out[2], "multi": out[3]}

    def render(self, idx=None, height: int = 600, width: int = 800, out: torch.Tensor | None = None) -> torch.Tensor:
        """RGB images of envs drawn on the device (the picture of renderer.scene()): a uint8 CUDA tensor
        (n, height, width, 3), written on the current stream.  Each image shows the state get_states() returns.

        idx: None (all envs), a host sequence / ndarray of env indices (checked here: ValueError), or an int64 CUDA
        tensor (not checked on the host: an out-of-range index gives an all-zero image).  out: an optional
        preallocated contiguous uint8 tensor of that shape on the sim's device, so that the call allocates nothing
        and can be captured in a CUDA graph."""
        idx, n = self._index(idx)
        dptr = None if idx is None else idx.data_ptr()
        shape = (n, int(height), int(width), 3)
        if out is None:
            out = torch.empty(shape, dtype=torch.uint8, device=self.device)
        elif tuple(out.shape) != shape or out.dtype != torch.uint8 or out.device != self.device or not out.is_contiguous():
            raise ValueError(f"out must be a contiguous uint8 tensor of shape {shape} on {self.device}")
        _capi.check(self._L.msoc_render(self._h, dptr, n, int(height), int(width), out.data_ptr(), self._stream()))
        return out

    def save_states(self, idx=None, out: torch.Tensor | None = None) -> torch.Tensor:
        """msoc_env_state records of envs as a (n, 808) uint8 CUDA tensor, written on the current stream without a host
        wait (the bytes of get_states; _capi.state_fields() gives named views).  idx as in render(): None (all envs), a
        host sequence (checked: ValueError), or an int64 CUDA tensor (not checked: an out-of-range index gives an
        all-zero record, whose hist_valid is 0).  out: an optional preallocated (n, 808) uint8 tensor on the sim's
        device, so that the call allocates nothing and can be captured in a CUDA graph."""
        idx, n = self._index(idx)
        shape = (n, _capi.ENV_STATE_BYTES)
        if out is not None and (tuple(out.shape) != shape or out.dtype != torch.uint8 or out.device != self.device):
            raise ValueError(f"out must be a uint8 tensor of shape {shape} on {self.device}")
        dst = out
        if out is None or not out.is_contiguous() or out.data_ptr() % 16:
            dst = torch.empty(shape, dtype=torch.uint8, device=self.device)
        _capi.check(self._L.msoc_save_states(self._h, None if idx is None else idx.data_ptr(), n, dst.data_ptr(),
                                             self._stream()))
        if out is not None and dst is not out:  # a misaligned or strided `out` gets a copy
            out.copy_(dst)
        return out if out is not None else dst

    def load_states(self, idx, states: torch.Tensor) -> None:
        """Installs msoc_env_state records (n, 808) uint8 (save_states(), or built with _capi.state_fields()) into the
        envs idx, on the current stream, with the semantics of set_states.  idx: None (envs 0..n-1), a host sequence
        (checked: ValueError when out of range or repeated), or an int64 CUDA tensor (not checked: out-of-range entries
        are skipped, repeated destinations are undefined).  The observation buffer is not written.  The first load on a
        sim allocates a side array (the records of injected states), so it cannot be the first call inside a CUDA graph
        capture.  A graph captured on this sim BEFORE that first load (or set_states) keeps stepping without the side
        array: load (or set_states) once before capturing any graph on a sim whose states you will load."""
        if not isinstance(states, torch.Tensor):
            states = torch.from_numpy(np.ascontiguousarray(states).view(np.uint8).reshape(-1, _capi.ENV_STATE_BYTES))
        if states.dim() != 2 or states.shape[1] != _capi.ENV_STATE_BYTES or states.dtype != torch.uint8:
            raise ValueError(f"states must be a (n, {_capi.ENV_STATE_BYTES}) uint8 tensor")
        idx, n = self._index(idx, unique=True, n_all=states.shape[0])
        if n != states.shape[0]:
            raise ValueError(f"{n} indices for {states.shape[0]} states")
        if n > self.num_envs and idx is None:
            raise ValueError(f"{n} states for {self.num_envs} envs")
        if states.device != self.device or not states.is_contiguous() or states.data_ptr() % 16:
            states = states.to(self.device).contiguous()
            if states.data_ptr() % 16:
                states = states.clone()
        _capi.check(self._L.msoc_load_states(self._h, None if idx is None else idx.data_ptr(), n, states.data_ptr(),
                                             self._stream()))

    def clone_envs(self, src, dst) -> None:
        """Env dst[k] becomes a copy of env src[k]: its state (save_states of src, then load_states) and its row of the
        observation buffer.  src is snapshot before anything is written, so src and dst may overlap and src may
        repeat; dst must not repeat.  Host index lists are checked (ValueError).  CUDA index tensors are not: a pair
        with either index out of range is skipped, as load_states skips such entries, without a host wait."""
        src_t, n = self._index(src)
        dst_t, m = self._index(dst, unique=True)
        if src is None or dst is None or n != m:
            raise ValueError("src and dst must be index lists of the same length")
        if n == 0:
            return
        N = self.num_envs
        valid = (src_t >= 0) & (src_t < N) & (dst_t >= 0) & (dst_t < N)
        snap = self.save_states(src_t)
        # Observation rows, with torch indexing, which needs every index in range: a skipped pair repeats the copy of
        # the first valid pair (the same bytes to the same row), or copies row 0 onto itself when no pair is valid.
        j = torch.argmax(valid.to(torch.uint8)).view(1)
        any_valid = valid.index_select(0, j)
        src_r = torch.where(valid, src_t, torch.where(any_valid, src_t.index_select(0, j), 0))
        dst_r = torch.where(valid, dst_t, torch.where(any_valid, dst_t.index_select(0, j), 0))
        rows = self.obs.index_select(0, src_r)
        self.load_states(torch.where(valid, dst_t, -1), snap)
        self.obs.index_copy_(0, dst_r, rows)

    STATE_FORMAT = "marl_soccer_b200.env_states/1"

    def state_dict(self) -> dict:
        """Everything needed to resume this sim exactly: every env's state (save_states()), the observation buffer (the
        policy's next input, which the states do not determine), the 8 statistics accumulators, and what the states
        are only valid for (config, env count, global env offset).  Tensors are copies on the sim's device.  The
        outputs of the last step (reward, done, goal, score) are not part of it."""
        return {"format": self.STATE_FORMAT, "num_envs": self.num_envs, "global_env_offset": self.global_env_offset,
                "config": json.loads(json.dumps(self.config)), "states": self.save_states(),
                "obs": self.obs.clone(), "stats": self._stats_live.clone()}

    def load_state_dict(self, d: dict) -> None:
        """Restores a state_dict() of a sim with the same env count, global env offset and config (ValueError
        otherwise; load_states moves env states between differently shaped sims)."""
        if d.get("format") != self.STATE_FORMAT:
            raise ValueError(f"not a {self.STATE_FORMAT} state dict: format {d.get('format')!r}")
        for key, mine in (("num_envs", self.num_envs), ("global_env_offset", self.global_env_offset),
                          ("config", json.loads(json.dumps(self.config)))):
            if d.get(key) != mine:
                raise ValueError(f"state dict {key} {d.get(key)!r} does not match this sim's {mine!r}")
        states, obs, stats = d["states"], d["obs"], d["stats"]
        if tuple(states.shape) != (self.num_envs, _capi.ENV_STATE_BYTES) or tuple(obs.shape) != tuple(self.obs.shape) \
                or tuple(stats.shape) != (8,):
            raise ValueError("state dict tensors do not have this sim's shapes")
        self.load_states(None, states)
        self.obs.copy_(obs)
        self._stats_live.copy_(stats)

    def get_states(self, idx) -> list:
        idx = np.ascontiguousarray(idx, dtype=np.int64)
        arr = (_capi.MsocEnvState * len(idx))()
        torch.cuda.synchronize(self.device)
        _capi.check(self._L.msoc_get_state(self._h, idx.ctypes.data, len(idx), C.byref(arr)))
        return list(arr)

    def set_states(self, idx, states) -> None:
        idx = np.ascontiguousarray(idx, dtype=np.int64)
        arr = (_capi.MsocEnvState * len(idx))(*states)
        torch.cuda.synchronize(self.device)
        _capi.check(self._L.msoc_set_state(self._h, idx.ctypes.data, len(idx), C.byref(arr)))

    def counters(self):
        """(score (N,2) int32, steps (N,) int32) of the live episodes, on the host."""
        score = np.zeros((self.num_envs, 2), np.int32)
        steps = np.zeros((self.num_envs,), np.int32)
        _capi.check(self._L.msoc_read_counters(self._h, score.ctypes.data, steps.ctypes.data, self._stream()))
        return score, steps
