"""Device-resident rollout half of the reference's PPO trainer (marl-soccer.ipynb:366-431) -- the immediate
caller of the hot path (SURVEY.md section 8f rank 1, BASELINE config 5).

Everything the notebook does around `envs.step` per rollout step stays on the GPU: observation normalisation
`clip((x - mean) / (std + 1e-8), -10, 10)` (:385), the policy/value MLPs (:125-190), action sampling, uniform
random actions for the red agents (:397-400), reward / done / value / log-prob storage (:403-409), and the
running mean/variance update (:264-296, :431).  The simulator is `BatchedSoccerSim` (one fused CUDA kernel per
step); nothing crosses PCIe inside the loop.  The network architecture and the normaliser arithmetic mirror
the reference so that its checkpoints (`runs/*/ppo_pettingzoo_soccer.ppo_model`,
`latest_normalizer_stats.npz`) load unchanged.
"""
from __future__ import annotations

import numpy as np
import torch
import torch.nn as nn
from torch.distributions.normal import Normal

from . import _capi


def layer_init(layer, std=np.sqrt(2), bias_const=0.0):
    torch.nn.init.orthogonal_(layer.weight, std)
    torch.nn.init.constant_(layer.bias, bias_const)
    return layer


class Agent(nn.Module):
    """Actor / critic MLPs 66 -> 512 -> 256 -> 128 -> 64 -> (3 | 1), tanh (marl-soccer.ipynb:125-190; same
    parameter names, so `load_state_dict` of a reference checkpoint works)."""

    def __init__(self, obs_dim: int = 66, act_dim: int = 3, rpo_alpha: float = 0.0):
        super().__init__()
        self.critic = nn.Sequential(
            layer_init(nn.Linear(obs_dim, 512)), nn.Tanh(), nn.Linear(512, 256), nn.Tanh(), nn.Linear(256, 128), nn.Tanh(),
            layer_init(nn.Linear(128, 64)), nn.Tanh(), layer_init(nn.Linear(64, 1), std=1.0))
        self.actor_mean = nn.Sequential(
            layer_init(nn.Linear(obs_dim, 512)), nn.Tanh(), nn.Linear(512, 256), nn.Tanh(), nn.Linear(256, 128), nn.Tanh(),
            layer_init(nn.Linear(128, 64)), nn.Tanh(), layer_init(nn.Linear(64, act_dim), std=0.01))
        self.actor_logstd = nn.Parameter(torch.zeros(1, act_dim))
        self.rpo_alpha = rpo_alpha

    def get_value(self, x):
        return self.critic(x)

    def get_action_and_value(self, x, action=None):
        mean = self.actor_mean(x)
        std = torch.exp(self.actor_logstd.expand_as(mean))
        probs = Normal(mean, std, validate_args=False)  # (validation syncs with the host: not capturable)
        if action is None:
            action = mean + std * torch.randn_like(mean)  # = probs.sample(), without torch.normal's host-side std check
        elif self.rpo_alpha > 0.0:
            z = torch.empty_like(mean).uniform_(-self.rpo_alpha, self.rpo_alpha)
            probs = Normal(mean + z, std, validate_args=False)
        return action, probs.log_prob(action).sum(1), probs.entropy().sum(1), self.critic(x)

    def get_deterministic_action(self, x):
        return self.actor_mean(x)


class RunningMeanStd:
    """Welford running mean / variance over a stream of observation batches, float64 on the device
    (marl-soccer.ipynb:264-296)."""

    def __init__(self, shape, device):
        self.mean = torch.zeros(shape, dtype=torch.float64, device=device)
        self.var = torch.ones(shape, dtype=torch.float64, device=device)
        self.count = 0

    def update(self, x: torch.Tensor) -> None:
        x = x.reshape(-1, self.mean.shape[-1]).to(torch.float64)
        batch_var, batch_mean = torch.var_mean(x, dim=0, unbiased=False)  # one Welford pass
        self.update_from_moments(batch_mean, batch_var, x.shape[0])

    def update_from_moments(self, batch_mean: torch.Tensor, batch_var: torch.Tensor, n: int) -> None:
        """Parallel-variance merge of one batch given by its mean, biased variance and size (marl-soccer.ipynb:275-296)."""
        batch_mean, batch_var = batch_mean.to(torch.float64), batch_var.to(torch.float64)
        delta = batch_mean - self.mean
        tot = self.count + n
        self.mean = self.mean + delta * (n / tot)
        m2 = self.var * self.count + batch_var * n + delta.square() * (self.count * n / tot)
        self.var = m2 / tot
        self.count = tot

    @property
    def std(self):
        return self.var.sqrt()

    def load_npz(self, path: str) -> None:
        z = np.load(path)
        self.mean = torch.as_tensor(z["mean"], dtype=torch.float64, device=self.mean.device)
        self.var = torch.as_tensor(z["var"], dtype=torch.float64, device=self.mean.device)

    def normalize(self, x: torch.Tensor) -> torch.Tensor:
        return torch.clamp((x - self.mean.float()) / (self.std.float() + 1e-8), -10.0, 10.0)


class EpisodeReturns:
    """One team's finished episodes and the sum of their returns, kept on the device the way msoc_stats keeps blue's
    (episodes, episode_return_sum): `running` (N,) fp32 is each env's return so far in its current episode, `sums` (2,)
    fp64 the episodes finished and their returns summed, since the last read(reset=True).  An episode that was already
    running when counting began is counted from there."""

    def __init__(self, num_envs: int, device):
        self.running = torch.zeros((num_envs,), device=device)
        self.sums = torch.zeros((2,), dtype=torch.float64, device=device)

    def add(self, reward: torch.Tensor, done: torch.Tensor) -> None:
        """One step: reward (N,) of the team, done (N,) of the same step (the truncation reward is the episode's last)."""
        d = done.to(torch.float32)
        self.running.add_(reward)
        self.sums[0].add_(d.sum())
        self.sums[1].add_((self.running * d).sum(dtype=torch.float64))
        self.running.mul_(1.0 - d)

    def read(self, reset: bool = False) -> dict:
        out = dict(zip(("episodes", "episode_return_sum"), self.sums.tolist()))
        if reset:
            self.sums.zero_()
        return out


class RolloutBuffer:
    """(T, N, A, ...) storage of one rollout for the A trainable agents, on the device.  agents=2: the blue agents.
    agents=4: self-play, one policy for both teams (collect_rollout / GraphedRollout with self_play=True).  Rows 2, 3
    are red's in the policy's frame: observations mirrored (selfplay.mirror_frames), actions as the policy returned
    them (red played their mirror_actions), so that log-probs and PPO ratios are those of the policy; log-probs,
    values, rewards (red's own, msoc_step_teams) and dones likewise.  `red_returns` (EpisodeReturns) then counts red's
    finished episodes and returns over the rollouts that use this buffer; blue's are in the sim's statistics."""

    def __init__(self, num_steps: int, num_envs: int, device, obs_dtype=torch.float32, agents: int = 2):
        if agents not in (2, 4):
            raise ValueError("agents must be 2 (blue) or 4 (both teams, self-play)")
        T, N, A = num_steps, num_envs, agents
        self.agents = A
        self.obs = torch.zeros((T, N, A, 66), dtype=obs_dtype, device=device)
        self.actions = torch.zeros((T, N, A, 3), device=device)
        self.logprobs = torch.zeros((T, N, A), device=device)
        self.rewards = torch.zeros((T, N, A), device=device)
        self.dones = torch.zeros((T, N, A), device=device)
        self.values = torch.zeros((T, N, A), device=device)
        self.red_returns = EpisodeReturns(N, device) if A == 4 else None


class PackedPolicy:
    """Inference-only packing of an `Agent`'s two MLPs for the rollout loop -- the same layers in `dtype` (bf16) with
    fp32 accumulation, laid out for the tensor cores (what the plain modules cost per step at 524 288 rows, under ncu, in
    brackets):
      * the first layer of both nets is ONE GEMM over inputs padded from 66 to 72 features (rows of 16-byte multiples;
        with K = 66 cuBLAS falls back to a legacy mma.sync kernel [0.5 ms per net]);
      * the hidden and output layers of the two nets are batched GEMMs over a (2, rows, width) stack: half the launches,
        one tanh pass per layer instead of two;
      * biases ride in the GEMMs: every layer's output has 8 extra channels, the first of which is the constant 1
        (tanh of a pre-activation of 20), and the next layer's weight matrix carries its bias in that column -- a batched
        GEMM has no bias epilogue, and `baddbmm` materialises the broadcast bias with a strided copy [0.8 ms].
    `refresh()` re-reads the agent's parameters (call it after every optimiser step).
    critic=False packs the actor alone (a stack of one net, for a policy whose value nobody reads: a frozen opponent);
    the calls then return None for the value."""

    IN = 72
    PAD = 8       # extra channels per layer: [1, 0, 0, 0, 0, 0, 0, 0]
    ONE = 20.0    # tanh(20) == 1 in fp32 and bf16

    def __init__(self, agent: Agent, dtype=torch.bfloat16, critic: bool = True):
        self.agent, self.dtype, self.critic = agent, dtype, critic
        dev = agent.actor_logstd.device
        P, S = self.PAD, 2 if critic else 1
        self.w0 = torch.zeros((S * (512 + P), self.IN), dtype=dtype, device=dev)
        self.b0 = torch.zeros((S * (512 + P),), dtype=dtype, device=dev)
        # hidden layers 512 -> 256 -> 128 -> 64 (each + PAD in and out), output layer 64 + PAD -> 8
        self.w = [torch.zeros((S, o + P, i + P), dtype=dtype, device=dev) for o, i in ((256, 512), (128, 256), (64, 128))]
        self.w.append(torch.zeros((S, 8, 64 + P), dtype=dtype, device=dev))
        self.refresh()

    @torch.no_grad()
    def refresh(self) -> None:
        P = self.PAD
        nets = (self.agent.actor_mean, self.agent.critic) if self.critic else (self.agent.actor_mean,)
        for k, net in enumerate(nets):
            base = (512 + P) * k
            self.w0[base:base + 512, :66].copy_(net[0].weight)
            self.b0[base:base + 512].copy_(net[0].bias)
            self.b0[base + 512] = self.ONE                       # the constant-1 channel of the first layer's output
            for j, layer in enumerate((2, 4, 6, 8)):
                wgt, bias = net[layer].weight, net[layer].bias
                o, i = wgt.shape
                self.w[j][k, :o, :i].copy_(wgt)
                self.w[j][k, :o, i].copy_(bias)                  # bias column: multiplies the constant-1 channel
                if j < 3:
                    self.w[j][k, o, i] = self.ONE                # this layer's own constant-1 channel

    @torch.no_grad()
    def __call__(self, x72: torch.Tensor):
        """x72: (rows, 72) normalised observations in `dtype`, columns 66.. zero.  Returns (mean (rows, 3), value (rows, 1)) fp32
        (value None without the critic)."""
        rows = x72.shape[0]
        h = torch.addmm(self.b0, x72, self.w0.t()).tanh_()           # (rows, 2 * 520) = [actor 512 + 8 | critic 512 + 8]
        h = h.view(rows, self.w0.shape[0] // (512 + self.PAD), 512 + self.PAD).transpose(0, 1)  # (2, rows, 520), strided: no copy
        for j in range(3):
            h = torch.bmm(h, self.w[j].transpose(1, 2)).tanh_()
        out = torch.bmm(h, self.w[3].transpose(1, 2))                  # (2, rows, 8)
        return out[0, :, :3].float(), out[1, :, :1].float() if self.critic else None

    @torch.no_grad()
    def act(self, x72: torch.Tensor):
        """Sampled action, its log-probability and the value (Agent.get_action_and_value with action=None)."""
        mean, value = self(x72)
        logstd = self.agent.actor_logstd.float().expand_as(mean)
        std = logstd.exp()
        noise = torch.randn_like(mean)
        action = mean + std * noise
        logprob = (-0.5 * noise.square() - logstd - 0.9189385332046727).sum(1)  # log N(a; mean, std), a = mean + std z
        return action, logprob, value


def _team_rows(obs: torch.Tensor) -> torch.Tensor:
    """(N, A, 66) rows -> (A N, 66) policy rows, team-major: [blue agents 0, 1 of every env | red agents 2, 3]."""
    n, A = obs.shape[0], obs.shape[1]
    if A == 2:
        return obs.reshape(-1, 66)
    return obs.reshape(n, 2, 2, 66).transpose(0, 1).reshape(-1, 66)


def _per_env(x: torch.Tensor, n: int, A: int) -> torch.Tensor:
    """Team-major policy outputs (A N, ...) -> (N, A, ...) (the inverse of _team_rows)."""
    rest = x.shape[1:]
    if A == 2:
        return x.reshape(n, 2, *rest)
    return x.reshape(2, n, 2, *rest).transpose(0, 1).reshape(n, 4, *rest)


def _check_self_play(buf, self_play: bool, opponent) -> None:
    if self_play and opponent is not None:
        raise ValueError("self_play trains red with the same policy: it cannot also play an opponent")
    if buf.obs.shape[2] != (4 if self_play else 2):
        raise ValueError("self_play needs RolloutBuffer(agents=4); without it the buffer has 2 agents")


def _policy_step(agent, x, policy_dtype):
    if policy_dtype is not None:
        with torch.autocast(device_type="cuda", dtype=policy_dtype):
            action, logprob, _, value = agent.get_action_and_value(x)
        return action.float(), logprob.float(), value.float()
    action, logprob, _, value = agent.get_action_and_value(x)
    return action, logprob, value


@torch.no_grad()
def collect_rollout(sim, agent: Agent, normalizer: RunningMeanStd, buf: RolloutBuffer, next_obs: torch.Tensor,
                    next_done: torch.Tensor, generator=None, update_normalizer: bool = True, policy_dtype=None,
                    deterministic: bool = False, opponent=None, self_play: bool = False):
    """One rollout of `buf.obs.shape[0]` steps (marl-soccer.ipynb:366-431): blue = policy, red = U(-1, 1), or red = the
    frozen snapshots of `opponent` (selfplay.Opponent; it samples or plays its mean as it was built to, whatever
    `deterministic` says).  Without self_play, red's observations never reach the buffer or the normaliser.
    next_obs: (N, 2, 66) raw observations of the blue agents (may be a view of the simulator's observation buffer: it is
    consumed before the next step overwrites it); next_done: (N, 2).  Returns the updated pair (next_obs is a view of
    sim.obs).  policy_dtype: optional autocast dtype for the MLPs (e.g. torch.bfloat16); the simulator is always fp32.
    deterministic: blue plays the policy mean and red stands still (eval.py:84-104 style; used by the parity test).
    self_play: one policy plays all four agents and learns from both teams (buf = RolloutBuffer(agents=4)): red's rows
    are mirrored into the policy's frame (selfplay.team_view), red plays mirror_actions of the policy's actions, and
    the step is msoc_step_teams, so red gets its own reward.  next_obs is then (N, 4, 66) in the policy's frame
    (selfplay.team_view(sim.obs)) and next_done (N, 4); the returned next_obs is a new tensor.  Red's observations
    enter the normaliser with blue's.  With deterministic=True both teams play the policy mean."""
    _check_self_play(buf, self_play, opponent)
    T, A = buf.obs.shape[0], buf.obs.shape[2]
    n = sim.num_envs
    full = sim.actions  # (N, 4, 3) device buffer of the handle
    mean32, inv_std32 = normalizer.mean.float(), 1.0 / (normalizer.std.float() + 1e-8)  # fp32 on the hot loop
    if self_play:
        from .selfplay import mirror_actions, team_view
    for t in range(T):
        buf.obs[t] = next_obs
        buf.dones[t] = next_done
        x = torch.clamp((_team_rows(next_obs) - mean32) * inv_std32, -10.0, 10.0)
        if deterministic:
            action = agent.get_deterministic_action(x)
            logprob, value = torch.zeros(x.shape[0], device=x.device), agent.get_value(x)
        else:
            action, logprob, value = _policy_step(agent, x, policy_dtype)
        buf.values[t] = _per_env(value, n, A).reshape(n, A)
        buf.actions[t] = _per_env(action, n, A)
        buf.logprobs[t] = _per_env(logprob, n, A)
        full[:, :2] = buf.actions[t, :, :2]
        if self_play:
            full[:, 2:] = mirror_actions(buf.actions[t, :, 2:])
        elif opponent is not None:
            opponent.act(sim)
        elif deterministic:
            full[:, 2:] = 0.0
        else:
            full[:, 2:].uniform_(-1.0, 1.0, generator=generator)
        obs, reward, done, _goal = sim.step(full, auto_reset=True, team_rewards=self_play)
        buf.rewards[t] = reward
        if self_play:
            buf.red_returns.add(reward[:, 2], done)
            next_obs = team_view(obs)
        else:
            next_obs = obs[:, :2]  # a view: read by the next iteration (or the caller) before the simulator steps again
        next_done = done.to(torch.float32)[:, None].expand(n, A)
    if update_normalizer:
        normalizer.update(buf.obs.reshape(-1, 66))
    return next_obs, next_done


class GraphedRollout:
    """collect_rollout as ONE CUDA graph per rollout: the T steps (normalise -> MLPs -> sample -> red actions ->
    msoc_step's two kernels -> storage) are captured once and replayed, so the ~30 launches per step cost no host
    time and the simulator is never waiting for Python.  The simulator's step counter lives in device memory, which
    is what makes a captured sequence of steps replayable (include/msoc.h).  Sampling uses torch's default CUDA
    generator (graph-safe).  A sim whose states will be loaded (load_states, load_state_dict, clone_envs, set_states)
    needs one such load before the graph is captured (include/msoc.h, msoc_load_states).
    opponent: a selfplay.Opponent plays red inside the graph instead of U(-1, 1); Opponent.set() writes a new snapshot
    into the buffers the graph reads, so the next replay plays it without a new capture.
    self_play: collect_rollout(self_play=True) as a graph (buf = RolloutBuffer(agents=4)): per step, blue's and red's
    mirrored rows (msoc_team_inputs, teams 0 and 1, on the fused bf16 path; selfplay.mirror_frames otherwise) form one
    (4N, 72) policy input, the policy runs once over it, red's actions are mirrored back into sim.actions[:, 2:] and
    the step is msoc_step_teams.  The normaliser's moments cover both teams.  run() then returns next_obs (N, 4, 66) in
    the policy's frame and next_done (N, 4)."""

    def __init__(self, sim, agent: Agent, normalizer: RunningMeanStd, buf: RolloutBuffer, policy_dtype=None,
                 update_normalizer: bool = True, opponent=None, self_play: bool = False):
        _check_self_play(buf, self_play, opponent)
        self.sim, self.agent, self.normalizer, self.buf, self.opponent = sim, agent, normalizer, buf, opponent
        self.policy_dtype, self.update_normalizer, self.self_play = policy_dtype, update_normalizer, self_play
        A = buf.obs.shape[2]
        dev = sim.device
        self.mean32 = torch.zeros((66,), device=dev)
        self.inv_std32 = torch.ones((66,), device=dev)
        self.shift32 = torch.zeros((66,), device=dev)  # -mean / (std + 1e-8)
        self.next_done = torch.zeros((sim.num_envs, A), device=dev)
        self.graph = None
        # bf16 policy: the packed form of the two MLPs and its padded input / fp32 staging buffers
        self.packed = PackedPolicy(agent, policy_dtype) if policy_dtype is not None else None
        if self.packed is not None:
            rows = sim.num_envs * A
            self.x32 = torch.empty((rows, 66), device=dev)
            self.x72 = torch.zeros((rows, PackedPolicy.IN), dtype=policy_dtype, device=dev)
        # per-step sums and sums of squares of the raw observations, gathered inside the graph; the running statistics merge
        # them in fp64 after the rollout -- instead of a float64 pass over the whole (T, N, 2, 66) buffer
        T = buf.obs.shape[0]
        self.moments = torch.zeros((T, 2, 66), dtype=torch.float64, device=dev)
        # bf16 policy + bf16 buffer: the three consumers of the observation rows are served by one kernel of the library
        self.fused_inputs = self.packed is not None and policy_dtype == torch.bfloat16 and buf.obs.dtype == torch.bfloat16
        self._L = _capi.lib() if self.fused_inputs else None
        if self.fused_inputs and self_play:  # the raw rows of the two teams, team-major, before they go to the buffer
            self.raw2 = torch.zeros((2, sim.num_envs, 2, 66), dtype=buf.obs.dtype, device=dev)

    def _refresh(self):
        self.mean32.copy_(self.normalizer.mean.float())
        self.inv_std32.copy_(1.0 / (self.normalizer.std.float() + 1e-8))
        self.shift32.copy_(-self.mean32 * self.inv_std32)
        if self.packed is not None:
            self.packed.refresh()

    @torch.no_grad()
    def _body(self):
        if self.self_play:
            return self._body_self_play()
        sim, buf, n = self.sim, self.buf, self.sim.num_envs
        full = sim.actions
        self.moments.zero_()
        for t in range(buf.obs.shape[0]):
            cur = sim.obs[:, :2]  # the blue agents' rows of the simulator's own buffer: no clone
            buf.dones[t] = self.next_done
            if self.fused_inputs:
                # one pass over the rows (msoc_policy_inputs): normalised + clipped + padded bf16 policy input, the raw
                # bf16 copy for the buffer, per-feature sum / sum of squares for the running normaliser
                _capi.check(self._L.msoc_policy_inputs(sim.obs.data_ptr(), n, self.shift32.data_ptr(), self.inv_std32.data_ptr(),
                                                       self.x72.data_ptr(), buf.obs[t].data_ptr(),
                                                       self.moments[t].data_ptr() if self.update_normalizer else None,
                                                       torch.cuda.current_stream(sim.device).cuda_stream))
            else:
                buf.obs[t] = cur
                if self.update_normalizer:  # the step's moments in fp32 (Welford), merged in fp64 after the rollout
                    v, m = torch.var_mean(cur.reshape(-1, 66), dim=0, unbiased=False)
                    self.moments[t, 0].copy_(m * (2 * n))
                    self.moments[t, 1].copy_((v + m.square()) * (2 * n))
                if self.packed is not None:
                    torch.addcmul(self.shift32, cur.reshape(-1, 66), self.inv_std32, out=self.x32)
                    self.x32.clamp_(-10.0, 10.0)
                    self.x72[:, :66].copy_(self.x32)
            if self.packed is not None:
                action, logprob, value = self.packed.act(self.x72)
            else:
                x = torch.clamp((cur.reshape(-1, 66) - self.mean32) * self.inv_std32, -10.0, 10.0)
                action, logprob, value = _policy_step(self.agent, x, self.policy_dtype)
            buf.values[t] = value.reshape(n, 2)
            buf.actions[t] = action.reshape(n, 2, 3)
            buf.logprobs[t] = logprob.reshape(n, 2)
            full[:, :2] = buf.actions[t]
            if self.opponent is not None:
                self.opponent.act(sim)
            else:
                full[:, 2:].uniform_(-1.0, 1.0)
            _obs, reward, done, _goal = sim.step(full, auto_reset=True)
            buf.rewards[t] = reward
            self.next_done.copy_(done.to(torch.float32)[:, None].expand(n, 2))

    def _body_self_play(self):
        from .selfplay import mirror_actions, mirror_frames
        sim, buf, n = self.sim, self.buf, self.sim.num_envs
        full = sim.actions
        stream = torch.cuda.current_stream(sim.device).cuda_stream
        self.moments.zero_()
        for t in range(buf.obs.shape[0]):
            buf.dones[t] = self.next_done
            if self.fused_inputs:
                # one pass per team (msoc_team_inputs; team 1 mirrors red's rows): rows [0, 2N) of the policy input are
                # blue's, [2N, 4N) red's; raw rows to the buffer; moments of both teams into the same sums
                for team in (0, 1):
                    _capi.check(self._L.msoc_team_inputs(sim.obs.data_ptr(), n, team, self.shift32.data_ptr(),
                                                         self.inv_std32.data_ptr(), self.x72[2 * n * team:].data_ptr(),
                                                         self.raw2[team].data_ptr(),
                                                         self.moments[t].data_ptr() if self.update_normalizer else None,
                                                         stream))
                buf.obs[t].view(n, 2, 2, 66).copy_(self.raw2.transpose(0, 1))
            else:
                rows = torch.cat([sim.obs[:, :2], mirror_frames(sim.obs[:, 2:])], 1)  # (N, 4, 66), the policy's frame
                buf.obs[t] = rows
                x = _team_rows(rows)
                if self.update_normalizer:
                    v, m = torch.var_mean(x, dim=0, unbiased=False)
                    self.moments[t, 0].copy_(m * (4 * n))
                    self.moments[t, 1].copy_((v + m.square()) * (4 * n))
                if self.packed is not None:
                    torch.addcmul(self.shift32, x, self.inv_std32, out=self.x32)
                    self.x32.clamp_(-10.0, 10.0)
                    self.x72[:, :66].copy_(self.x32)
            if self.packed is not None:
                action, logprob, value = self.packed.act(self.x72)
            else:
                x = torch.clamp((x - self.mean32) * self.inv_std32, -10.0, 10.0)
                action, logprob, value = _policy_step(self.agent, x, self.policy_dtype)
            buf.values[t] = _per_env(value, n, 4).reshape(n, 4)
            buf.actions[t] = _per_env(action, n, 4)
            buf.logprobs[t] = _per_env(logprob, n, 4)
            full[:, :2] = buf.actions[t, :, :2]
            full[:, 2:] = mirror_actions(buf.actions[t, :, 2:])
            _obs, reward, done, _goal = sim.step(full, auto_reset=True, team_rewards=True)
            buf.rewards[t] = reward
            buf.red_returns.add(reward[:, 2], done)
            self.next_done.copy_(done.to(torch.float32)[:, None].expand(n, 4))

    def run(self):
        """One rollout; returns (next_obs view, next_done)."""
        self._refresh()
        dev = self.sim.device
        if self.graph is None:
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                self._body()  # eager warm-up on the capture stream (cuBLAS workspaces, autocast caches)
            torch.cuda.current_stream(dev).wait_stream(side)
            torch.cuda.synchronize(dev)
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph, stream=side):
                self._body()
        else:
            self.graph.replay()
        if self.update_normalizer:
            count = self.moments.shape[0] * self.sim.num_envs * self.buf.obs.shape[2]
            total = self.moments.sum(0)
            mean = total[0] / count
            self.normalizer.update_from_moments(mean, total[1] / count - mean.square(), count)
        if self.self_play:
            from .selfplay import team_view
            return team_view(self.sim.obs), self.next_done
        return self.sim.obs[:, :2], self.next_done


@torch.no_grad()
def compute_gae(agent: Agent, normalizer: RunningMeanStd, buf: RolloutBuffer, next_obs, next_done, gamma=0.995,
                gae_lambda=0.95):
    """Generalised advantage estimation over the rollout (marl-soccer.ipynb:454-464), for any number of agents A per env
    (buf.rewards (T, N, A); next_obs (N, A, 66), next_done (N, A))."""
    T, n, A = buf.rewards.shape
    next_value = agent.get_value(normalizer.normalize(next_obs.reshape(-1, 66))).reshape(n, A)
    adv = torch.zeros_like(buf.rewards)
    last = torch.zeros((n, A), device=buf.rewards.device)
    for t in reversed(range(T)):
        nonterminal = 1.0 - (next_done if t == T - 1 else buf.dones[t + 1])
        nv = next_value if t == T - 1 else buf.values[t + 1]
        delta = buf.rewards[t] + gamma * nv * nonterminal - buf.values[t]
        last = delta + gamma * gae_lambda * nonterminal * last
        adv[t] = last
    return adv, adv + buf.values
