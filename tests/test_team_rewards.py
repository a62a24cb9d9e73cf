"""Red's own reward (msoc_step_teams, env_step's TEAMS instances) and the shared-policy self-play rollout, without a GPU:
the host harness's red column against an fp64 restatement of the definition (include/msoc.h) and against blue's reward
of the mirrored state, blue's outputs bit for bit those of the plain step, the argument checks, the agents=4 buffer and
compute_gae."""
import ctypes as C
from types import SimpleNamespace

import numpy as np
import pytest
import torch

import parity_util as P
from hostsim_lib import HostSim
from hostsim_teams_lib import TeamsHostSim
from selfplay_util import mirror_state
from marl_soccer_b200 import _capi, build
from marl_soccer_b200.rollout import (Agent, EpisodeReturns, GraphedRollout, RolloutBuffer, RunningMeanStd,
                                      collect_rollout, compute_gae)
from marl_soccer_b200.selfplay import mirror_actions, team_view

CFG = P.CONFIG
KINDS = ("open", "walls", "scrum", "goal")


def _band(a, b):
    """worst |a - b| / (atol + rtol |b|) of the reward band (DESIGN.md section 3)"""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.max(np.abs(a - b) / (P.ATOL["reward"] + P.RTOL * np.abs(b))))


def _states(n, seed):
    """all four kinds; every fifth state one step from truncation"""
    rng = np.random.default_rng(seed)
    max_steps = CFG["simulation"]["max_steps"]
    out = []
    for i in range(n):
        s = P.random_state(rng, KINDS[i % 4])
        if i % 5 == 0:
            s["steps"] = max_steps - 1
        out.append(s)
    return out


def _harness(states, cls=TeamsHostSim, seed=0):
    h = cls(len(states), CFG, seed=seed)
    for i, s in enumerate(states):
        h.set_state(i, P.oracle_to_dev_state(s))
    return h


def _red_reward_fp64(pre, goal, post_score, post_steps):
    """include/msoc.h's red column in fp64 from the pre-step state (positions, velocities, bias velocities: the step's
    displacement), the step's goal flag and the post-step score and step count."""
    rw = CFG["rewards"]
    pos = np.array(pre.pos, np.float64)
    inc = (np.array(pre.vel, np.float64) + np.array(pre.vbias, np.float64)) / 60.0

    def drop(d, l):
        return np.hypot(*d) - np.hypot(*(d + l))

    r = 0.0
    if rw["ball_proximity_multiplier"] != 0.0:
        r += rw["ball_proximity_multiplier"] * sum(drop(pos[i] - pos[4], inc[i] - inc[4]) for i in (2, 3))
    r += rw["move_ball_to_goal_multiplier"] * drop(pos[4] - np.array([10.0, 300.0]), inc[4])
    if goal < 0:
        r += rw["goal_scored_reward"]
    if goal > 0:
        r -= rw["goal_conceded_penalty"]
    r -= rw["alive_penalty"]
    if post_steps >= CFG["simulation"]["max_steps"]:
        r = rw["score_difference_multiplier"] * (post_score[1] - post_score[0])
    return r


def test_red_column_is_the_definition_and_blue_is_untouched():
    """768 injected states (open field, walls, scrums, goal mouths; every fifth one step from truncation), two steps of
    the harness with red's reward (the first from the injected records, which the general path steps; the second
    through every work class): the red column equals an fp64 restatement of the definition within the reward band;
    every other output, and the states after each step, are those of the plain step bit for bit."""
    n = 768
    states = _states(n, 31)
    rng = np.random.default_rng(32)
    teams, plain = _harness(states), _harness(states, HostSim)  # plain: the blue-only harness (hostsim.cu, hsim_step)
    worst, goals_b, goals_r, truncs, classes, contacts = 0.0, 0, 0, 0, set(), 0
    for _ in range(2):
        act = rng.uniform(-1.2, 1.2, (n, 4, 3)).astype(np.float32)
        pre = [teams.get_state(i) for i in range(n)]
        o_t, r_t, d_t, g_t = teams.step(act, auto_reset=False, team_rewards=True)
        c, load = teams.last()
        o_p, r_p, d_p, g_p = plain.step(act, auto_reset=False)
        assert r_t.shape == (n, 4)
        assert r_t[:, :2].tobytes() == r_p.tobytes()
        assert o_t.tobytes() == o_p.tobytes() and np.array_equal(d_t, d_p) and np.array_equal(g_t, g_p)
        assert np.array_equal(teams.score, plain.score)
        assert np.array_equal(r_t[:, 2], r_t[:, 3])
        post = [teams.get_state(i) for i in range(n)]
        for i in range(n):
            assert bytes(post[i]) == bytes(plain.get_state(i)), i
        assert teams.stats() == plain.stats()
        want = np.array([_red_reward_fp64(pre[i], int(g_t[i]), tuple(post[i].score), post[i].steps) for i in range(n)])
        worst = max(worst, _band(r_t[:, 2], want))
        goals_b, goals_r, truncs = goals_b + int((g_t > 0).sum()), goals_r + int((g_t < 0).sum()), truncs + int(d_t.sum())
        classes |= {int(k) for k in load}
        contacts += int(c.sum())
    P.record("team_rewards_definition_hostsim", {"envs": n, "steps": 2, "worst_violation_ratio": round(worst, 3),
                                                 "goals_blue": goals_b, "goals_red": goals_r, "truncations": truncs,
                                                 "classes": sorted(classes)})
    assert goals_b > 0 and goals_r > 0 and truncs >= n // 5
    assert {-1, 0, 1, 2, 3} <= classes and contacts > 0  # contact-free and all four contact classes
    assert worst <= 1.0, worst


def test_red_reward_of_s_is_blue_reward_of_the_mirrored_state():
    """One harness holds S in envs [0, n) and M(S) in [n, 2n), stepped with (b, r) and (M(r), M(b)): red's reward of S
    equals blue's of M(S) within the reward band on every env (goal steps and truncations included; envs whose ball
    lands within rounding of a goal plane are left out, as in every goal comparison), and the other way round."""
    n = 512
    states = _states(n, 41)
    mirrored = [mirror_state(s) for s in states]
    rng = np.random.default_rng(42)
    act = rng.uniform(-1.2, 1.2, (n, 4, 3)).astype(np.float32)
    act_m = np.concatenate([mirror_actions(act[:, 2:]), mirror_actions(act[:, :2])], axis=1)
    h = _harness(states + mirrored)
    _, r, d, g = h.step(np.concatenate([act, act_m]), auto_reset=False, team_rewards=True)
    keep = ~(P.goal_knife_edge(states) | P.goal_knife_edge(mirrored))
    assert np.array_equal(d[:n], d[n:]) and np.array_equal(g[:n][keep], -g[n:][keep])
    worst = max(_band(r[:n, 2][keep], r[n:, 0][keep]), _band(r[:n, 0][keep], r[n:, 2][keep]))
    goals = g[:n][keep]
    P.record("team_rewards_mirror_hostsim", {"pairs": n, "compared": int(keep.sum()), "worst_violation_ratio": round(worst, 3),
                                             "goal_steps": int((goals != 0).sum()), "truncations": int(d[:n].sum())})
    assert (goals > 0).sum() > 0 and (goals < 0).sum() > 0 and d[:n].sum() > 0
    assert worst <= 1.0, worst


def test_step_teams_rejects_bad_arguments_without_a_device():
    L = C.CDLL(build.build())
    _capi.declare(L)
    buf = (C.c_float * 64)()
    p = C.c_void_p(C.addressof(buf))
    assert L.msoc_step_teams(None, p, p, p, p, p, None, 0, None) == -1
    assert b"msoc_step_teams" in L.msoc_last_error()
    for k in range(5):  # each required pointer NULL in turn (the handle is checked first, so it is NULL here too)
        args = [p] * 5
        args[k] = None
        assert L.msoc_step_teams(None, *args, None, 0, None) == -1
    assert "msoc_step_teams" in _capi.EXPORTS


def test_self_play_buffer_shapes_and_argument_checks():
    buf = RolloutBuffer(3, 5, "cpu", agents=4)
    assert buf.obs.shape == (3, 5, 4, 66) and buf.actions.shape == (3, 5, 4, 3)
    for t in (buf.logprobs, buf.rewards, buf.dones, buf.values):
        assert t.shape == (3, 5, 4)
    assert buf.red_returns.running.shape == (5,) and buf.red_returns.sums.dtype == torch.float64
    two = RolloutBuffer(3, 5, "cpu")
    assert two.obs.shape == (3, 5, 2, 66) and two.red_returns is None and two.agents == 2
    with pytest.raises(ValueError):
        RolloutBuffer(3, 5, "cpu", agents=3)
    agent, rms = Agent(), RunningMeanStd((66,), "cpu")
    sim = SimpleNamespace(num_envs=5, device=torch.device("cpu"))
    with pytest.raises(ValueError):  # self-play and an opponent
        collect_rollout(sim, agent, rms, buf, None, None, self_play=True, opponent=object())
    with pytest.raises(ValueError):  # self-play needs the 4-agent buffer
        collect_rollout(sim, agent, rms, two, None, None, self_play=True)
    with pytest.raises(ValueError):  # and the 4-agent buffer needs self-play
        collect_rollout(sim, agent, rms, buf, None, None)
    with pytest.raises(ValueError):
        GraphedRollout(sim, agent, rms, buf, self_play=True, opponent=object())
    with pytest.raises(ValueError):
        GraphedRollout(sim, agent, rms, two, self_play=True)


def test_team_view_mirrors_red_rows_only():
    x = np.random.default_rng(3).normal(size=(6, 4, 66)).astype(np.float32)
    v = team_view(x)
    from marl_soccer_b200.selfplay import mirror_frames
    assert v[:, :2].tobytes() == x[:, :2].tobytes() and v[:, 2:].tobytes() == mirror_frames(x[:, 2:]).tobytes()
    assert torch.equal(team_view(torch.from_numpy(x)), torch.from_numpy(v))


def test_episode_returns_counts_finished_episodes():
    er = EpisodeReturns(3, "cpu")
    for r, d in (([1.0, 2.0, 3.0], [0, 1, 0]), ([0.5, 0.25, -1.0], [1, 0, 0]), ([1.0, 1.0, 1.0], [0, 1, 1])):
        er.add(torch.tensor(r), torch.tensor(d, dtype=torch.uint8))
    # env 0: 1 + 0.5 at step 2; env 1: 2 at step 1, 0.25 + 1 at step 3; env 2: 3 - 1 + 1 at step 3
    assert er.read(reset=True) == {"episodes": 4.0, "episode_return_sum": 1.5 + 2.0 + 1.25 + 3.0}
    assert er.read() == {"episodes": 0.0, "episode_return_sum": 0.0}
    assert er.running.tolist() == [1.0, 0.0, 0.0]


def _gae_two_agents(agent, normalizer, buf, next_obs, next_done, gamma=0.995, gae_lambda=0.95):
    """compute_gae as it was for the two blue agents only (the parent's code)"""
    T, n = buf.rewards.shape[0], buf.rewards.shape[1]
    next_value = agent.get_value(normalizer.normalize(next_obs.reshape(-1, 66))).reshape(n, 2)
    adv = torch.zeros_like(buf.rewards)
    last = torch.zeros((n, 2), device=buf.rewards.device)
    for t in reversed(range(T)):
        nonterminal = 1.0 - (next_done if t == T - 1 else buf.dones[t + 1])
        nv = next_value if t == T - 1 else buf.values[t + 1]
        delta = buf.rewards[t] + gamma * nv * nonterminal - buf.values[t]
        last = delta + gamma * gae_lambda * nonterminal * last
        adv[t] = last
    return adv, adv + buf.values


def _seeded(buf, g):
    buf.rewards.copy_(torch.randn(buf.rewards.shape, generator=g))
    buf.values.copy_(torch.randn(buf.values.shape, generator=g))
    buf.dones.copy_((torch.rand(buf.dones.shape, generator=g) < 0.1).float())


def test_compute_gae_two_agents_bit_identical_and_four_agents_per_column():
    torch.manual_seed(0)
    agent, rms = Agent(), RunningMeanStd((66,), "cpu")
    g = torch.Generator().manual_seed(5)
    T, n = 9, 7
    two = RolloutBuffer(T, n, "cpu")
    _seeded(two, g)
    nxt, nd = torch.randn((n, 2, 66), generator=g), (torch.rand((n, 2), generator=g) < 0.2).float()
    with torch.no_grad():
        adv, ret = compute_gae(agent, rms, two, nxt, nd)
        adv0, ret0 = _gae_two_agents(agent, rms, two, nxt, nd)
    assert adv.numpy().tobytes() == adv0.numpy().tobytes() and ret.numpy().tobytes() == ret0.numpy().tobytes()
    # four agents: the two halves of the buffer are two independent 2-agent problems
    four = RolloutBuffer(T, n, "cpu", agents=4)
    _seeded(four, g)
    nxt4, nd4 = torch.randn((n, 4, 66), generator=g), (torch.rand((n, 4), generator=g) < 0.2).float()
    with torch.no_grad():
        adv4, ret4 = compute_gae(agent, rms, four, nxt4, nd4)
        for h in (0, 1):
            half = RolloutBuffer(T, n, "cpu")
            for k in ("rewards", "values", "dones"):
                getattr(half, k).copy_(getattr(four, k)[:, :, 2 * h:2 * h + 2])
            a, r = compute_gae(agent, rms, half, nxt4[:, 2 * h:2 * h + 2], nd4[:, 2 * h:2 * h + 2])
            assert torch.allclose(adv4[:, :, 2 * h:2 * h + 2], a, atol=1e-6) and torch.allclose(ret4[:, :, 2 * h:2 * h + 2], r, atol=1e-6)
