"""Red's own reward on the device (msoc_step_teams) and the shared-policy self-play rollout: a teams handle against a
plain one over a long run (every output but red's column bit for bit), red's column against the host harness and
against blue's reward of the mirrored state, graph replay, the general path and the checked build, and the self-play
rollout (eager against a host loop, graphed against an eager re-run of what it stored)."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import parity_util as P
from hostsim_teams_lib import TeamsHostSim
from selfplay_util import mirror_state
from marl_soccer_b200 import _capi
from marl_soccer_b200.rollout import Agent, GraphedRollout, RolloutBuffer, RunningMeanStd, collect_rollout
from marl_soccer_b200.selfplay import mirror_actions, mirror_frames, team_view
from marl_soccer_b200.sim import BatchedSoccerSim

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _band(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.max(np.abs(a - b) / (P.ATOL["reward"] + P.RTOL * np.abs(b)))) if a.size else 0.0


def _cfg(max_steps):
    return {**P.CONFIG, "simulation": {"max_steps": max_steps}}


def test_teams_handle_matches_the_plain_handle_step_for_step():
    """4 096 envs, two handles with the same seed and actions, 240 steps with auto-reset (max_steps 60): obs, done,
    goal, score, reward columns 0, 1, saved states and statistics of msoc_step_teams equal msoc_step's bit for bit;
    the run has goals for both sides, truncations and every contact class."""
    n, steps = 4096, 240
    a, b = (BatchedSoccerSim(n, config=_cfg(60), device=DEV, seed=3) for _ in range(2))
    for s in (a, b):
        s.reset(_capi.MODE_FULL_RANDOM, seed=9)
    g = torch.Generator(device=DEV).manual_seed(1)
    classes = np.zeros(4, np.int64)
    goals_b = goals_r = truncs = 0
    for t in range(steps):
        act = torch.rand((n, 4, 3), generator=g, device=DEV) * 2.4 - 1.2
        o_a, r_a, d_a, g_a = a.step(act)
        o_b, r_b, d_b, g_b = b.step(act, team_rewards=True)
        assert r_b.shape == (n, 4) and r_b is b.reward4
        assert torch.equal(o_a, o_b) and torch.equal(d_a, d_b) and torch.equal(g_a, g_b), t
        assert torch.equal(a.score, b.score) and torch.equal(r_a, r_b[:, :2]), t
        assert torch.equal(r_b[:, 2], r_b[:, 3]) and bool(torch.isfinite(r_b).all()), t
        classes += np.array(list(b.class_counts().values()))
        goals_b += int((g_b > 0).sum())
        goals_r += int((g_b < 0).sum())
        truncs += int(d_b.sum())
    assert torch.equal(a.save_states(), b.save_states())
    sa, sb = a.stats(), b.stats()  # the fp64 return sum is added with atomics, in no fixed order
    assert sa.pop("episode_return_sum") == pytest.approx(sb.pop("episode_return_sum"), rel=1e-6)
    assert sa == sb
    P.record("team_rewards_side_by_side", {"envs": n, "steps": steps, "goals_blue": goals_b, "goals_red": goals_r,
                                           "truncations": truncs, "classes_light_heavy_pair_multi": classes.tolist()})
    assert goals_b > 0 and goals_r > 0 and truncs >= n and (classes > 0).all(), (goals_b, goals_r, truncs, classes)


def test_red_column_against_the_harness_and_the_mirrored_state():
    """S in envs [0, n) and M(S) in [n, 2n) of one handle and of the host harness (states of all four kinds, every
    fifth one step from truncation), one step with (b, r) and (M(r), M(b)): the device's four reward columns equal the
    harness's within the reward band, and red's reward of S equals blue's of M(S) (goal planes' rounding cases left
    out)."""
    n = 1024
    rng = np.random.default_rng(51)
    states = []
    for i in range(n):
        s = P.random_state(rng, P.KINDS[i % 4])
        if i % 5 == 0:
            s["steps"] = P.CONFIG["simulation"]["max_steps"] - 1
        states.append(s)
    mirrored = [mirror_state(s) for s in states]
    act = rng.uniform(-1.2, 1.2, (n, 4, 3)).astype(np.float32)
    act_m = np.concatenate([mirror_actions(act[:, 2:]), mirror_actions(act[:, :2])], axis=1)
    full = np.concatenate([act, act_m])
    recs = [P.oracle_to_dev_state(s) for s in states + mirrored]
    sim = BatchedSoccerSim(2 * n, config=P.CONFIG, device=DEV, seed=1)
    arr = np.frombuffer(b"".join(bytes(r) for r in recs), np.uint8).reshape(2 * n, _capi.ENV_STATE_BYTES)
    sim.load_states(None, torch.from_numpy(arr.copy()))
    _, r, d, g = sim.step(torch.from_numpy(full).to(DEV), auto_reset=False, team_rewards=True)
    r, d, g = r.cpu().numpy(), d.cpu().numpy(), g.cpu().numpy()
    h = TeamsHostSim(2 * n, P.CONFIG, seed=1)
    for i, rec in enumerate(recs):
        h.set_state(i, rec)
    _, r_h, d_h, g_h = h.step(full, auto_reset=False, team_rewards=True)
    keep = ~(P.goal_knife_edge(states) | P.goal_knife_edge(mirrored))
    keep2 = np.concatenate([keep, keep])
    assert np.array_equal(d, d_h) and np.array_equal(g[keep2], g_h[keep2])
    w_h = _band(r[keep2], r_h[keep2])
    w_m = max(_band(r[:n, 2][keep], r[n:, 0][keep]), _band(r[:n, 0][keep], r[n:, 2][keep]))
    P.record("team_rewards_device_references", {"pairs": n, "compared": int(keep.sum()), "vs_harness": round(w_h, 3),
                                                "vs_mirrored_blue": round(w_m, 3), "goal_steps": int((g[:n] != 0).sum()),
                                                "truncations": int(d[:n].sum())})
    assert (g[:n][keep] > 0).any() and (g[:n][keep] < 0).any() and d[:n].sum() > 0
    assert w_h <= 1.0 and w_m <= 1.0, (w_h, w_m)


def _run(n, steps, seed):
    """rewards (steps, n, 4) of a seeded team-reward run, and the sim and actions for a replay"""
    sim = BatchedSoccerSim(n, config=_cfg(25), device=DEV, seed=seed)
    sim.reset(_capi.MODE_FULL_RANDOM, seed=seed)
    g = torch.Generator(device=DEV).manual_seed(seed)
    acts = [torch.rand((n, 4, 3), generator=g, device=DEV) * 2.4 - 1.2 for _ in range(steps)]
    snap = sim.state_dict()
    sim.load_state_dict(snap)  # every run starts from loaded records, as the replay below does
    out = []
    for a in acts:
        out.append(sim.step(a, team_rewards=True)[1].clone())
    return torch.stack(out), sim, acts, snap


@pytest.mark.parametrize("n", [1, 33, 70001])
def test_graph_replay_and_general_path_give_the_eager_rewards(n):
    steps = 30
    eager, sim, acts, snap = _run(n, steps, 5)
    # a captured step, replayed with each step's actions
    sim.load_state_dict(snap)
    static = torch.zeros_like(acts[0])
    side = torch.cuda.Stream(device=DEV)
    side.wait_stream(torch.cuda.current_stream(DEV))
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=side):
        sim.step(static, team_rewards=True)
    for t, a in enumerate(acts):
        static.copy_(a)
        graph.replay()
        assert torch.equal(sim.reward4, eager[t]), (n, t)
    # every contact through the general path, from states re-synchronised every step (the two paths contract their
    # contact arithmetic differently, which free-running steps would amplify; tests/test_gpu_parity.py does the same)
    gen = BatchedSoccerSim(n, config=_cfg(25), device=DEV, seed=5)
    worst = 0.0
    for a in acts:
        gen.load_states(None, sim.save_states())
        r = sim.step(a, team_rewards=True)[1].clone()
        _, r_g, d_g, g_g = gen.step(a, team_rewards=True, general_path=True)
        assert torch.equal(d_g, sim.done) and torch.equal(g_g, sim.goal)
        worst = max(worst, _band(r_g.cpu().numpy(), r.cpu().numpy()))
    assert worst <= 1.0, worst


CHECKED = r"""
import sys
sys.path.insert(0, %(root)r); sys.path.insert(0, %(root)r + "/tests")
import torch
from marl_soccer_b200 import _capi
from marl_soccer_b200.sim import BatchedSoccerSim
import parity_util as P
L = _capi.lib()
assert L.msoc_debug_errors() == 0
for n in (1, 33, 70001):
    sim = BatchedSoccerSim(n, config={**P.CONFIG, "simulation": {"max_steps": 25}}, device="cuda:0", seed=5)
    sim.reset(2, seed=5)
    sim.load_state_dict(sim.state_dict())
    g = torch.Generator(device="cuda:0").manual_seed(5)
    acts = [torch.rand((n, 4, 3), generator=g, device="cuda:0") * 2.4 - 1.2 for _ in range(30)]
    rs = torch.stack([sim.step(a, team_rewards=True)[1].clone() for a in acts])
    assert L.msoc_debug_errors() == 0, n
    torch.save(rs.cpu(), %(tmp)r + f"/checked_{n}.pt")
print("checked teams clean")
"""


def test_checked_build_runs_the_team_instances(tmp_path):
    from marl_soccer_b200 import build
    env = dict(os.environ, MSOC_LIB=build.build_checked())
    r = subprocess.run([sys.executable, "-c", CHECKED % {"root": ROOT, "tmp": str(tmp_path)}], env=env,
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "checked teams clean" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]
    for n in (1, 33, 70001):
        eager = _run(n, 30, 5)[0].cpu()
        assert _band(torch.load(tmp_path / f"checked_{n}.pt").numpy(), eager.numpy()) <= 1.0, n


def _agent(seed):
    torch.manual_seed(seed)
    a = Agent()
    with torch.no_grad():
        for p in a.parameters():
            p.add_(0.05 * torch.randn_like(p))
    r = RunningMeanStd((66,), DEV)
    r.mean = torch.randn(66, dtype=torch.float64, device=DEV) * 0.1
    r.var = torch.rand(66, dtype=torch.float64, device=DEV) + 0.5
    return a.to(DEV), r


def test_deterministic_self_play_rollout_matches_a_host_loop():
    """collect_rollout(self_play=True, deterministic=True) against the loop it stands for: red's input built with
    mirror_frames, the agent's mean for all four rows, red's actions mirrored back, red's reward from the teams step."""
    n, T = 512, 40
    agent, rms = _agent(3)
    sims = [BatchedSoccerSim(n, config=_cfg(15), device=DEV, seed=2) for _ in range(2)]
    for s in sims:
        s.reset(_capi.MODE_FULL_RANDOM, seed=4)
    buf = RolloutBuffer(T, n, DEV, agents=4)
    obs0 = team_view(sims[0].obs)
    nxt, nd = collect_rollout(sims[0], agent, rms, buf, obs0, torch.zeros((n, 4), device=DEV),
                              update_normalizer=False, deterministic=True, self_play=True)
    sim = sims[1]
    inv = 1.0 / (rms.std.float() + 1e-8)
    ret, red_eps, red_sum = torch.zeros(n, device=DEV), 0, 0.0
    for t in range(T):
        rows = torch.cat([sim.obs[:, :2], mirror_frames(sim.obs[:, 2:])], 1)
        assert torch.allclose(buf.obs[t], rows, atol=2e-4), t
        with torch.no_grad():  # the policy's rows team by team: blue's 2N, then red's mirrored 2N
            team_rows = torch.cat([rows[:, :2].reshape(-1, 66), rows[:, 2:].reshape(-1, 66)])
            x = torch.clamp((team_rows - rms.mean.float()) * inv, -10.0, 10.0)
            act = agent.actor_mean(x).view(2, n, 2, 3).transpose(0, 1).reshape(n, 4, 3)
            val = agent.get_value(x).view(2, n, 2).transpose(0, 1).reshape(n, 4)
        assert torch.allclose(buf.actions[t], act, atol=2e-4) and torch.allclose(buf.values[t], val, atol=2e-3), t
        full = torch.cat([act[:, :2], mirror_actions(act[:, 2:])], 1)
        _, r, d, _ = sim.step(full, team_rewards=True)
        assert torch.allclose(buf.rewards[t], r, atol=1e-5), t
        ret += r[:, 2]
        red_eps += int(d.sum())
        red_sum += float((ret * d.float()).sum())
        ret *= 1.0 - d.float()
    assert torch.allclose(nxt, team_view(sim.obs), atol=2e-4) and nd.shape == (n, 4)
    got = buf.red_returns.read()
    assert red_eps > 0 and got["episodes"] == red_eps and abs(got["episode_return_sum"] - red_sum) <= 1e-3 * max(1.0, abs(red_sum))


@pytest.mark.parametrize("dtype", [None, torch.bfloat16])
def test_graphed_self_play_rollout_matches_an_eager_rerun(dtype):
    """GraphedRollout(self_play=True) (fp32, and bf16 with the fused msoc_team_inputs path), one replay; then the sim is
    rewound and what the graph stored is re-run eagerly: red's stored rows are mirror_frames of the sim's rows 2, 3
    (blue's rows as they are), the stored actions (mirrored for red) step the sim to the stored rewards and dones bit
    for bit, and the values and log-probs are the agent's on the stored rows (fp32 within 1e-3, bf16 within the
    tolerances of DESIGN.md section 11)."""
    n, T = 4096, 16
    obs_dtype = torch.float32 if dtype is None else torch.bfloat16
    sim = BatchedSoccerSim(n, config=_cfg(10), device=DEV, seed=6)
    sim.reset(_capi.MODE_FULL_RANDOM, seed=6)
    agent, rms = _agent(8)
    buf = RolloutBuffer(T, n, DEV, obs_dtype=obs_dtype, agents=4)
    sim.load_state_dict(sim.state_dict())  # states will be loaded below: once before the capture
    ro = GraphedRollout(sim, agent, rms, buf, policy_dtype=dtype, self_play=True)
    ro.run()
    assert ro.graph is not None
    snap, done0 = sim.state_dict(), ro.next_done.clone()
    mean, inv = rms.mean.float().clone(), 1.0 / (rms.std.float() + 1e-8)
    count0 = rms.count
    nxt, _ = ro.run()  # a replay
    torch.cuda.synchronize()
    assert rms.count == count0 + T * n * 4
    assert torch.equal(nxt, team_view(sim.obs))
    sim.load_state_dict(snap)
    tol_v, tol_lp = (1e-3, 1e-3) if dtype is None else (5e-2, 1e-1)
    worst_v = worst_lp = 0.0
    done = done0
    for t in range(T):
        rows = team_view(sim.obs)
        assert torch.equal(buf.obs[t], rows.to(obs_dtype)), t
        assert torch.equal(buf.dones[t], done), t
        with torch.no_grad():
            x = torch.clamp((rows.reshape(-1, 66) - mean) * inv, -10.0, 10.0)
            _, lp, _, v = agent.get_action_and_value(x, buf.actions[t].reshape(-1, 3))
        worst_v = max(worst_v, float((v.view(n, 4) - buf.values[t]).abs().max()))
        worst_lp = max(worst_lp, float((lp.view(n, 4) - buf.logprobs[t]).abs().max()))
        full = torch.cat([buf.actions[t, :, :2], mirror_actions(buf.actions[t, :, 2:])], 1)
        _, r, d, _ = sim.step(full, team_rewards=True)
        assert torch.equal(buf.rewards[t], r), t
        done = d.float()[:, None].expand(n, 4)
    P.record(f"team_rewards_graphed_rollout_{'bf16' if dtype else 'fp32'}", {"envs": n, "steps": T,
                                                                            "worst_value": worst_v, "worst_logprob": worst_lp})
    assert worst_v < tol_v and worst_lp < tol_lp, (worst_v, worst_lp)
    assert buf.red_returns.read()["episodes"] > 0
