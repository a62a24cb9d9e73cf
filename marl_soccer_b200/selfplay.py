"""Self-play against frozen policy snapshots: red played by earlier versions of the blue policy.

The field is symmetric about x = 400 and red's observation frames are built from red's own side (include/msoc.h,
msoc_team_inputs), so a blue policy plays red unchanged when it sees red's frames mirrored and its actions are mirrored
back.  `mirror_frames` / `mirror_actions` are that transform (the reference implementation the CUDA kernel is tested
against, and the helpers for host users of SyncMultiAgentVecEnv / HostBufferSim who run their own red policy).
`Opponent` is a pool of frozen snapshots playing red in contiguous slices of the envs, inside collect_rollout /
GraphedRollout (rollout.py) or `evaluate_match`; red then gets no reward and only blue learns.  For one policy that
learns from both teams, collect_rollout / GraphedRollout take self_play=True instead (msoc_step_teams gives red its own
reward; `team_view` is the observation that policy sees).
"""
from __future__ import annotations

import numpy as np
import torch

from . import _capi
from .rollout import Agent, PackedPolicy, RunningMeanStd

FRAME, OBS = _capi.FRAME, _capi.OBS
# features of a 22-float frame whose sign the mirror flips: vx, omega and the x components of the five unit vectors
# (mate, opponent 0, opponent 1, ball, own goal, opponent goal); feature 2 (angle / pi) maps to the wrap of pi - theta
NEGATED = (0, 3, 4, 7, 10, 13, 16, 19)
ANGLE = 2
_NEG_SLICES = (slice(0, 1), slice(3, 4), slice(4, 20, 3))  # NEGATED as basic slices: no index tensor (graph-capturable)


def mirror_frames(x):
    """M applied to every 22-float frame of `x` (torch tensor or NumPy array, last dim 22 or 66, any leading dims): a red
    agent's frame becomes the frame a blue agent sees on the field mirrored about x = 400.  Negated: features 0, 3, 4,
    7, 10, 13, 16, 19; the angle feature a becomes 1 - a for a >= 0 (+0 and -0 included) and -1 - a otherwise, in the
    input's precision; the rest are unchanged.  Returns a new array of the same type, dtype and shape."""
    if x.shape[-1] not in (FRAME, OBS):
        raise ValueError(f"the last dimension must be {FRAME} or {OBS}, got {tuple(x.shape)}")
    if isinstance(x, np.ndarray):
        f = np.array(x, copy=True).reshape(*x.shape[:-1], -1, FRAME)
        a = f[..., ANGLE].copy()
        f[..., ANGLE] = np.where(a >= 0, 1 - a, -1 - a)
    else:
        f = x.clone().reshape(*x.shape[:-1], -1, FRAME)
        a = f[..., ANGLE].clone()
        f[..., ANGLE] = torch.where(a >= 0, 1 - a, -1 - a)
    for s in _NEG_SLICES:
        f[..., s] = -f[..., s]
    return f.reshape(x.shape)


def team_view(obs):
    """(N, 4, 66) observation rows -> the same rows in the frame of a policy that plays both teams (self-play): blue's
    rows 0, 1 as they are, red's rows 2, 3 mirrored (mirror_frames).  A new tensor or array."""
    if isinstance(obs, np.ndarray):
        return np.concatenate([obs[:, :2], mirror_frames(obs[:, 2:])], 1)
    return torch.cat([obs[:, :2], mirror_frames(obs[:, 2:])], 1)


def mirror_actions(a):
    """Mirror of actions (torch or NumPy, last dim 3): (a0, a1, a2) -> (a0, -a1, -a2).  World force = R(theta) (a0, a1)
    and torque a2, so under x -> 800 - x, theta -> pi - theta this is exact; clipping commutes with it."""
    if a.shape[-1] != 3:
        raise ValueError(f"the last dimension must be 3, got {tuple(a.shape)}")
    out = np.array(a, copy=True) if isinstance(a, np.ndarray) else a.clone()
    out[..., 1:] = -out[..., 1:]
    return out


class Opponent:
    """A pool of `slots` frozen policy snapshots that play red: slot k plays envs [k N // K, (k + 1) N // K).

    set(k, agent, normalizer) copies a blue Agent's parameters and its RunningMeanStd into slot k's own buffers, in
    place, so a GraphedRollout captured with this opponent plays the new snapshot on its next replay.  A slot plays an
    untrained Agent until it is set.  act(sim) writes red's actions of every env into sim.actions[:, 2:]: for slot k,
    mirror_actions(policy_k(clip(M(red rows) * inv_std_k + shift_k, -10, 10))), sampled with the snapshot's
    actor_logstd, or its mean when `deterministic`.

    policy_dtype None: the snapshot's fp32 modules.  torch.bfloat16 (CUDA only): per slot one msoc_team_inputs(team=1)
    pass (mirror, normalise, clip, bf16, pad) and an actor-only PackedPolicy; an opponent needs no value, so it pays for
    no critic."""

    def __init__(self, num_envs: int, slots: int = 1, device="cuda", policy_dtype=None, deterministic: bool = False):
        if slots < 1 or num_envs < 1:
            raise ValueError("an opponent needs at least one env and one slot")
        if policy_dtype not in (None, torch.bfloat16):
            raise ValueError("policy_dtype must be None (fp32) or torch.bfloat16")
        self.num_envs, self.slots, self.deterministic = int(num_envs), int(slots), bool(deterministic)
        self.device = torch.device(device)
        self.policy_dtype = policy_dtype
        self.bounds = [k * self.num_envs // self.slots for k in range(self.slots + 1)]
        with torch.random.fork_rng(devices=[]):  # the initial weights do not disturb the caller's random stream
            self.agents = [Agent().to(self.device).requires_grad_(False) for _ in range(self.slots)]
        self.shift = torch.zeros((self.slots, OBS), device=self.device)   # -mean / (std + 1e-8), fp32
        self.inv_std = torch.ones((self.slots, OBS), device=self.device)  # 1 / (std + 1e-8), fp32
        self.packed = None
        if policy_dtype is not None:
            if self.device.type != "cuda":
                raise ValueError("the bf16 opponent runs msoc_team_inputs: it needs a CUDA device")
            self._L = _capi.lib()
            self.packed = [PackedPolicy(a, policy_dtype, critic=False) for a in self.agents]
            self.x72 = torch.zeros((2 * self.num_envs, PackedPolicy.IN), dtype=policy_dtype, device=self.device)

    def slot_range(self, k: int) -> tuple[int, int]:
        return self.bounds[k], self.bounds[k + 1]

    @torch.no_grad()
    def set(self, k: int, agent: Agent, normalizer: RunningMeanStd) -> None:
        """Slot k becomes a frozen copy of `agent` with the observation normaliser `normalizer` (copied in place)."""
        if not 0 <= k < self.slots:
            raise IndexError(f"slot {k} of {self.slots}")
        self.agents[k].load_state_dict(agent.state_dict())
        inv = 1.0 / (normalizer.std.float().to(self.device) + 1e-8)
        self.inv_std[k].copy_(inv)
        self.shift[k].copy_(-normalizer.mean.float().to(self.device) * inv)
        if self.packed is not None:
            self.packed[k].refresh()

    @torch.no_grad()
    def act(self, sim) -> None:
        """Red's actions for the current observation: reads sim.obs (N, 4, 66) rows 2, 3, writes sim.actions[:, 2:]."""
        obs, actions = sim.obs, sim.actions
        if obs.shape[0] != self.num_envs:
            raise ValueError(f"this opponent was built for {self.num_envs} envs, the sim has {obs.shape[0]}")
        for k in range(self.slots):
            b0, b1 = self.slot_range(k)
            m = b1 - b0
            if m == 0:
                continue
            if self.packed is not None:
                x72 = self.x72[2 * b0:2 * b1]
                _capi.check(self._L.msoc_team_inputs(obs[b0].data_ptr(), m, 1, self.shift[k].data_ptr(),
                                                     self.inv_std[k].data_ptr(), x72.data_ptr(), None, None,
                                                     torch.cuda.current_stream(obs.device).cuda_stream))
                mean, _ = self.packed[k](x72)
            else:
                rows = mirror_frames(obs[b0:b1, 2:].reshape(-1, OBS))
                x = torch.clamp(torch.addcmul(self.shift[k], rows, self.inv_std[k]), -10.0, 10.0)
                mean = self.agents[k].actor_mean(x)
            if self.deterministic:
                action = mean
            else:
                action = mean + self.agents[k].actor_logstd.float().exp() * torch.randn_like(mean)
            actions[b0:b1, 2:] = mirror_actions(action.view(m, 2, 3))


@torch.no_grad()
def evaluate_match(sim, agent: Agent, normalizer: RunningMeanStd, opponent: Opponent, episodes: int = 1,
                   deterministic: bool = True, mode: int = _capi.MODE_FULL_RANDOM, seed: int | None = None,
                   reset: bool = True) -> list:
    """Blue (`agent` with `normalizer`) against every slot of `opponent`: resets all envs (msoc_reset in `mode`, seeded
    when `seed` is given), plays episodes * max_steps steps with auto-reset, and counts on the device, per slot, at every
    done: wins, draws and losses (the sign of the episode's final score blue - red) and goals for and against (blue's
    and red's final score).  Blue plays its mean when `deterministic`, else samples; red plays as `opponent` was built.
    The host waits once, at the end.  Returns one dict per slot.

    reset=False plays from the states the sim holds (e.g. a set of start states installed with load_states; the
    observation buffer is the policies' first input).  Every env should then be at step 0 of its episode, so that each
    of its `episodes` episodes is counted whole.

    This overwrites the sim's env states, observation buffer and statistics accumulators.  To continue training
    afterwards, wrap the call: `snap = sim.state_dict(); evaluate_match(...); sim.load_state_dict(snap)`."""
    n, K = sim.num_envs, opponent.slots
    if opponent.num_envs != n:
        raise ValueError(f"the opponent was built for {opponent.num_envs} envs, the sim has {n}")
    steps = int(episodes) * int(sim.config["simulation"]["max_steps"])
    dev = sim.device
    inv = 1.0 / (normalizer.std.float().to(dev) + 1e-8)
    shift = -normalizer.mean.float().to(dev) * inv
    counts = torch.zeros((n, 5), dtype=torch.int64, device=dev)  # wins, draws, losses, goals for, goals against
    if reset:
        sim.reset(mode, seed=seed)
    full = sim.actions
    for _ in range(steps):
        x = torch.clamp(torch.addcmul(shift, sim.obs[:, :2].reshape(-1, OBS), inv), -10.0, 10.0)
        mean = agent.actor_mean(x)
        act = mean if deterministic else mean + agent.actor_logstd.float().exp() * torch.randn_like(mean)
        full[:, :2] = act.view(n, 2, 3)
        opponent.act(sim)
        _obs, _rew, done, _goal = sim.step(full, auto_reset=True)
        score = sim.score.to(torch.int64)  # the episode's score, taken before the auto-reset
        diff = score[:, 0] - score[:, 1]
        outcome = torch.stack([diff > 0, diff == 0, diff < 0], 1).to(torch.int64)
        counts += done.to(torch.int64)[:, None] * torch.cat([outcome, score], 1)
    per_slot = torch.stack([counts[b0:b1].sum(0) for b0, b1 in (opponent.slot_range(k) for k in range(K))]).cpu()
    keys = ("wins", "draws", "losses", "goals_for", "goals_against")
    out = []
    for k in range(K):
        b0, b1 = opponent.slot_range(k)
        row = {"slot": k, "envs": b1 - b0, "episodes": int(episodes) * (b1 - b0)}
        row.update({key: int(v) for key, v in zip(keys, per_slot[k].tolist())})
        out.append(row)
    return out
