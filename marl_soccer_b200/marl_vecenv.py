"""Drop-in for the reference's `marl_vecenv.py` (soccer_simulation/marl_vecenv.py:3-79).

`SyncMultiAgentVecEnv(env_fns)` keeps the NumPy contract of the reference -- reset() -> (N,4,66) float32;
step((N,4,3)) -> obs (N,4,66) float32, rewards (N,4) float64 (columns 2,3 are zero), terminations (N,4)
bool (all False), truncations (N,4) bool, infos = sequence of N dicts keyed by agent -- but the Python
`for env in self.envs` loop (marl_vecenv.py:39) is one fused CUDA step (three kernel launches, DESIGN.md section 5) over all N
envs, including the auto-reset in full-random mode (marl_vecenv.py:45-53).

`TorchSoccerVecEnv` is the zero-copy variant for device-resident trainers: same semantics, torch CUDA
tensors in and out, infos only on demand.
"""
from __future__ import annotations

from typing import Optional

import numpy as np

from . import _capi
from .soccer_env import SoccerEnv, _AGENTS
from .spaces import Box


class LazyInfos:
    """Sequence of per-env info dicts ({agent: {"score": {...}, ["goal_scored_by": ...]}}), materialised
    per env on access from the step's score/goal snapshot (the reference builds N dicts every step)."""

    def __init__(self, score: np.ndarray, goal: np.ndarray):
        self._score, self._goal = score, goal

    def __len__(self):
        return int(self._goal.shape[0])

    def __getitem__(self, i):
        if isinstance(i, slice):
            return [self[k] for k in range(*i.indices(len(self)))]
        if i < 0:
            i += len(self)
        if not 0 <= i < len(self):
            raise IndexError(i)
        info = {"score": {"blue": int(self._score[i, 0]), "red": int(self._score[i, 1])}}
        g = int(self._goal[i])
        if g:
            info["goal_scored_by"] = "blue" if g > 0 else "red"
        return {a: dict(info) for a in _AGENTS}

    def __iter__(self):
        return (self[i] for i in range(len(self)))


class _EnvView:
    """Stand-in for one entry of `vec.envs` (the reference keeps N SoccerEnv objects there)."""

    def __init__(self, vec: "SyncMultiAgentVecEnv", index: int):
        self._vec, self.index = vec, index
        self.possible_agents = list(_AGENTS)

    def observation_space(self, agent):
        return self._vec.single_observation_space

    def action_space(self, agent):
        return self._vec.single_action_space

    def close(self):
        pass


class SyncMultiAgentVecEnv:
    def __init__(self, env_fns, *, num_envs: Optional[int] = None, config: Optional[dict] = None, seed: Optional[int] = None,
                 device: int = 0, global_env_offset: int = 0, pinned_buffers: bool = False, _sim_factory=None):
        """env_fns: list of callables as in the reference; only its length and (when `config` is not given)
        the config of env_fns[0]() are used -- N single-env CUDA handles would defeat the batching.
        Alternatively pass env_fns=None with num_envs / config.  pinned_buffers: one persistent set of page-locked host
        buffers (HostBufferSim(pinned=True)): full PCIe speed for large batches, but the arrays step() returns are then
        views that the next step overwrites."""
        if env_fns is not None:
            n = len(env_fns)
            if config is None:
                probe = env_fns[0]()
                config = getattr(probe, "_config", None)
                if hasattr(probe, "close"):
                    probe.close()
        else:
            n = int(num_envs)
        if config is None:
            from .sim import load_default_config
            config = load_default_config()
        self.num_envs = n
        self.config = config
        self.single_observation_space = Box(low=-np.inf, high=np.inf, shape=(66,), dtype=np.float32)
        self.single_action_space = Box(low=-1.0, high=1.0, shape=(3,), dtype=np.float32)
        self.possible_agents = list(_AGENTS)
        if seed is None:
            seed = int(np.random.SeedSequence().generate_state(1, dtype=np.uint64)[0] >> 1)
        if _sim_factory is None:
            from .host_api import HostBufferSim
            self._sim = HostBufferSim(n, config, seed=seed, global_offset=global_env_offset, device=device, pinned=pinned_buffers)
        else:
            self._sim = _sim_factory(n, config, seed)
        self.envs = [_EnvView(self, i) for i in range(n)]

    def reset(self, options=None, seed=None):
        """Resets all environments; env i is seeded with seed + i (marl_vecenv.py:23).  Returns only the
        stacked observations (N,4,66), like the reference."""
        use_fixed = use_full_random = False
        if isinstance(options, dict):
            use_fixed = bool(options.get("use_fixed_positions", False))
            use_full_random = bool(options.get("use_full_random_positions", False))
        mode = _capi.MODE_FIXED if use_fixed else _capi.MODE_FULL_RANDOM if use_full_random else _capi.MODE_RANDOM
        return self._sim.reset(mode, seed=None if seed is None else int(seed))

    def step(self, actions):
        actions = np.asarray(actions, dtype=np.float32)
        if actions.shape != (self.num_envs, 4, 3):
            raise ValueError(f"actions must have shape ({self.num_envs}, 4, 3), got {actions.shape}")
        if not np.all(np.isfinite(actions)):
            raise ValueError("Action contains non-finite values")  # soccer_env.py:116-117
        obs, rew, done, goal = self._sim.step(actions, auto_reset=True)
        rewards = np.zeros((self.num_envs, 4), np.float64)
        rewards[:, :2] = rew
        terms = np.zeros((self.num_envs, 4), bool)
        truncs = np.repeat(done.astype(bool)[:, None], 4, axis=1)
        return obs, rewards, terms, truncs, LazyInfos(self._sim.score.copy(), goal.copy())

    def render(self, idx=(0,), height: int = 600, width: int = 800) -> np.ndarray:
        """RGB images (len(idx), height, width, 3) uint8 of the envs `idx`, drawn on the GPU (HostBufferSim.render)."""
        return self._sim.render(idx, height, width)

    def _dict_to_array(self, data_dict):
        return np.array([data_dict[a] for a in self.possible_agents])

    def _array_to_dict(self, data_array):
        return {a: data_array[i] for i, a in enumerate(self.possible_agents)}

    def close(self):
        if hasattr(self._sim, "close"):
            self._sim.close()


class TorchSoccerVecEnv:
    """Device-resident vector env: torch CUDA tensors in and out, nothing crosses PCIe.

    step(actions (N,4,3) float32 cuda) -> obs (N,4,66) f32, rewards (N,2) f32 [blue agents; the (N,4)
    layout of the NumPy class with its two zero columns is available as `rewards4()`], truncations (N,)
    bool, goal (N,) int8.  Buffers are views valid until the next step."""

    def __init__(self, num_envs: int, config: Optional[dict] = None, device="cuda:0", seed: int = 0,
                 global_env_offset: int = 0):
        from .sim import BatchedSoccerSim
        self.sim = BatchedSoccerSim(num_envs, config=config, device=device, seed=seed,
                                    global_env_offset=global_env_offset)
        self.num_envs = int(num_envs)
        self.possible_agents = list(_AGENTS)
        self.single_observation_space = Box(low=-np.inf, high=np.inf, shape=(66,), dtype=np.float32)
        self.single_action_space = Box(low=-1.0, high=1.0, shape=(3,), dtype=np.float32)

    def reset(self, options=None, seed=None):
        use_fixed = bool(options.get("use_fixed_positions", False)) if isinstance(options, dict) else False
        use_full = bool(options.get("use_full_random_positions", False)) if isinstance(options, dict) else False
        mode = _capi.MODE_FIXED if use_fixed else _capi.MODE_FULL_RANDOM if use_full else _capi.MODE_RANDOM
        return self.sim.reset(mode, seed=seed)

    def step(self, actions, team_rewards: bool = False):
        """team_rewards: rewards (N,4) f32 with red's own reward in columns 2, 3 (BatchedSoccerSim.step)."""
        obs, rew, done, goal = self.sim.step(actions, auto_reset=True, team_rewards=team_rewards)
        return obs, rew, done.bool(), goal

    def rewards4(self):
        import torch
        r = torch.zeros((self.num_envs, 4), dtype=torch.float32, device=self.sim.device)
        r[:, :2] = self.sim.reward
        return r

    def render(self, idx=None, height: int = 600, width: int = 800, out=None):
        """RGB images (n, height, width, 3) uint8 on the device: BatchedSoccerSim.render."""
        return self.sim.render(idx, height, width, out)

    def state_dict(self) -> dict:
        """Env states, observation buffer and statistics: BatchedSoccerSim.state_dict."""
        return self.sim.state_dict()

    def load_state_dict(self, d: dict) -> None:
        self.sim.load_state_dict(d)

    def infos(self) -> LazyInfos:
        return LazyInfos(self.sim.score.cpu().numpy(), self.sim.goal.cpu().numpy())

    def close(self):
        self.sim.close()
