"""Self-play on the device: msoc_team_inputs against the reference mirror, a paired handle of S and M(S), the Opponent
(fp32 and bf16) against the blue policy on mirrored states, the Opponent inside a captured GraphedRollout, and
evaluate_match against a host loop."""
from types import SimpleNamespace

import numpy as np
import pytest
import torch

import oracle_lib as O
import parity_util as P
from selfplay_util import mirror_obs, mirror_state
from marl_soccer_b200 import _capi
from marl_soccer_b200.rollout import Agent, GraphedRollout, RolloutBuffer, RunningMeanStd
from marl_soccer_b200.selfplay import Opponent, evaluate_match, mirror_actions, mirror_frames
from marl_soccer_b200.sim import BatchedSoccerSim

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")


def _stream():
    return torch.cuda.current_stream(DEV).cuda_stream


def test_team_inputs_against_the_reference_mirror():
    L = _capi.lib()
    g = torch.Generator(device=DEV).manual_seed(4)
    for n in (1, 5, 1000, 70001):
        obs = torch.randn((n, 4, 66), generator=g, device=DEV) * 3.0
        obs[0, 2, :4] = torch.tensor([1e4, -1e4, 0.0, 1.0], device=DEV)  # clipped at +-10, the angle's edge cases
        obs[0, 3, 2], obs[0, 3, 24], obs[0, 3, 46] = -0.0, -1.0, 0.5
        obs0 = obs.clone()
        mean, std = torch.randn(66, generator=g, device=DEV), torch.rand(66, generator=g, device=DEV) + 0.5
        inv_std = 1.0 / (std + 1e-8)
        shift = -mean * inv_std
        x72 = torch.full((2 * n, 72), 7.0, dtype=torch.bfloat16, device=DEV)  # columns 66.. must stay untouched
        raw = torch.zeros((n, 2, 66), dtype=torch.bfloat16, device=DEV)
        mom = torch.zeros((2, 66), dtype=torch.float64, device=DEV)
        for _ in range(2):  # moments accumulate
            _capi.check(L.msoc_team_inputs(obs.data_ptr(), n, 1, shift.data_ptr(), inv_std.data_ptr(), x72.data_ptr(),
                                           raw.data_ptr(), mom.data_ptr(), _stream()))
        rows = mirror_frames(obs[:, 2:].reshape(-1, 66))
        ref = torch.clamp(torch.addcmul(shift, rows, inv_std), -10.0, 10.0).to(torch.bfloat16)
        assert torch.equal(x72[:, :66], ref) and bool((x72[:, 66:] == 7.0).all()), n
        assert torch.equal(raw, rows.view(n, 2, 66).to(torch.bfloat16)), n
        r64 = rows.to(torch.float64)
        assert torch.allclose(mom[0], 2 * r64.sum(0), rtol=1e-6, atol=1e-3) and torch.allclose(mom[1], 2 * r64.square().sum(0), rtol=1e-6)
        assert torch.equal(obs, obs0)
        # team 0 is msoc_policy_inputs: policy input and raw copy bit for bit; the fp64 moments are sums of per-block
        # partials added with atomics, whose order (and so the last bits) differs from launch to launch of either call
        outs = []
        for fn, args in ((L.msoc_policy_inputs, ()), (L.msoc_team_inputs, (0,))):
            x, r, m = torch.zeros_like(x72), torch.zeros_like(raw), torch.zeros_like(mom)
            _capi.check(fn(obs.data_ptr(), n, *args, shift.data_ptr(), inv_std.data_ptr(), x.data_ptr(), r.data_ptr(),
                           m.data_ptr(), _stream()))
            outs.append((x, r, m))
        (x_a, r_a, m_a), (x_b, r_b, m_b) = outs
        assert torch.equal(x_a, x_b) and torch.equal(r_a, r_b), n
        assert torch.allclose(m_a, m_b, rtol=1e-12, atol=1e-9), n
        # NULL raw / moments are skipped
        x = torch.zeros_like(x72)
        _capi.check(L.msoc_team_inputs(obs.data_ptr(), n, 1, shift.data_ptr(), inv_std.data_ptr(), x.data_ptr(), None, None, _stream()))
        assert torch.equal(x[:, :66], ref)


def _paired_sim(n, seed):
    """envs [0, n): states S (open, walls, goal kinds); envs [n, 2n): M(S); plus the oracle's contact-free mask of one
    step of both with random actions, and those actions (S's and the mirrored ones for M(S))."""
    rng = np.random.default_rng(seed)
    kinds = ("open", "walls", "goal")
    states = [P.random_state(rng, kinds[i % 3]) for i in range(n)]
    mirrored = [mirror_state(s) for s in states]
    sim = BatchedSoccerSim(2 * n, config=P.CONFIG, device=DEV, seed=1)
    recs = [P.oracle_to_dev_state(s) for s in states + mirrored]
    arr = np.frombuffer(b"".join(bytes(r) for r in recs), np.uint8).reshape(2 * n, _capi.ENV_STATE_BYTES)
    sim.load_states(None, torch.from_numpy(arr.copy()))
    act = rng.uniform(-1.2, 1.2, (n, 4, 3)).astype(np.float32)
    act_m = np.concatenate([mirror_actions(act[:, 2:]), mirror_actions(act[:, :2])], axis=1)
    ora, ora_m = O.OracleVec(n, P.CONFIG, seed=0), O.OracleVec(n, P.CONFIG, seed=0)
    ora.set_states(states)
    ora_m.set_states(mirrored)
    _, _, _, g = ora.step(act, auto_reset=False)
    ora_m.step(act_m, auto_reset=False)
    free = np.array([not (g[i] or ora.env(i).contact_count() or ora_m.env(i).contact_count()) for i in range(n)])
    free &= ~(P.goal_knife_edge(states) | P.goal_knife_edge(mirrored))
    return sim, act, act_m, free


def test_paired_handle_steps_through_the_mirror():
    """S in envs [0, n), M(S) in [n, 2n) of one handle, one step with mirrored actions: states and observations of the
    pairs are mirror images within the parity bands on every env the oracle finds contact-free and goal-free."""
    n = 1024
    sim, act, act_m, free = _paired_sim(n, 21)
    full = torch.from_numpy(np.concatenate([act, act_m])).to(DEV)
    obs, _, done, goal = sim.step(full, auto_reset=False)
    torch.cuda.synchronize()
    obs, done, goal = obs.cpu().numpy(), done.cpu().numpy(), goal.cpu().numpy()
    assert np.array_equal(done[:n], done[n:])
    st = sim.get_states(np.arange(2 * n))
    worst = {}
    for i in np.nonzero(free)[0]:
        a = P.dev_to_oracle_state(st[i], obs[i])
        b = P.dev_to_oracle_state(st[n + i], obs[n + i])
        assert a["score"] == b["score"][::-1] and a["steps"] == b["steps"]
        c = P.compare_state(mirror_state(dict(a, cache=[], obs=None)), b)
        c["obs"] = P.compare_obs(mirror_obs(obs[i]), obs[n + i])
        for k, v in c.items():
            worst[k] = max(worst.get(k, 0.0), v)
    P.record("selfplay_paired_handle", {"pairs": n, "compared": int(free.sum()),
                                        "worst_violation_ratio": {k: round(v, 3) for k, v in worst.items()}})
    assert free.sum() >= n // 4 and max(worst.values()) <= 1.0, worst


def _snapshot(seed):
    torch.manual_seed(seed)
    a = Agent()
    with torch.no_grad():
        for p in a.parameters():
            p.add_(0.1 * torch.randn_like(p))
    r = RunningMeanStd((66,), "cpu")
    r.mean = torch.randn(66, dtype=torch.float64) * 0.1
    r.var = torch.rand(66, dtype=torch.float64) + 0.5
    a = a.to(DEV)
    r.mean, r.var = r.mean.to(DEV), r.var.to(DEV)
    return a, r


@pytest.mark.parametrize("dtype", [None, torch.bfloat16])
def test_opponent_on_s_plays_what_blue_plays_on_the_mirrored_state(dtype):
    """Snapshot P plays red on S through Opponent; P plays blue on M(S) directly: red's actions on S are the mirror of
    blue's on M(S) (fp32 within 1e-3; the bf16 path within a recorded tolerance)."""
    n = 1024
    sim, act, act_m, free = _paired_sim(n, 22)
    sim.step(torch.from_numpy(np.concatenate([act, act_m])).to(DEV), auto_reset=False)  # observations from the step
    a, r = _snapshot(9)
    opp = Opponent(2 * n, slots=1, device=DEV, policy_dtype=dtype, deterministic=True)
    opp.set(0, a, r)
    opp.act(sim)
    inv = 1.0 / (r.std.float() + 1e-8)
    with torch.no_grad():
        x = torch.clamp(torch.addcmul(-r.mean.float() * inv, sim.obs[n:, :2].reshape(-1, 66), inv), -10.0, 10.0)
        blue_m = a.actor_mean(x).view(n, 2, 3)
    red = sim.actions[:n, 2:]
    f = torch.from_numpy(free).to(DEV)
    err = float((red[f] - mirror_actions(blue_m)[f]).abs().max())
    P.record(f"selfplay_opponent_vs_mirrored_blue_{'bf16' if dtype else 'fp32'}", {"pairs": int(free.sum()), "max_abs_error": err})
    assert err < (1e-3 if dtype is None else 5e-2), err


def _graphed(n, K, seed):
    cfg = dict(P.CONFIG)
    cfg["simulation"] = {"max_steps": 50}
    sim = BatchedSoccerSim(n, config=cfg, device=DEV, seed=seed)
    sim.reset(2, seed=seed)
    torch.manual_seed(seed)
    agent = Agent().to(DEV)
    rms = RunningMeanStd((66,), DEV)
    buf = RolloutBuffer(1, n, DEV, obs_dtype=torch.bfloat16)
    opp = Opponent(n, slots=K, device=DEV, policy_dtype=torch.bfloat16, deterministic=True)
    snaps = [_snapshot(seed + 10 + k) for k in range(K)]
    for k, (a, r) in enumerate(snaps):
        opp.set(k, a, r)
    ro = GraphedRollout(sim, agent, rms, buf, policy_dtype=torch.bfloat16, opponent=opp)
    ro.run()  # eager warm-up and capture
    return sim, opp, ro, snaps


def _replay_and_eager(sim, opp, ro):
    before = sim.obs.clone()
    ro.run()  # a replay of the captured graph
    torch.cuda.synchronize()
    red = sim.actions[:, 2:].clone()
    shadow = SimpleNamespace(obs=before, actions=torch.zeros_like(sim.actions))
    opp.act(shadow)
    return red, shadow.actions[:, 2:], before


def test_graphed_rollout_plays_the_opponent_and_picks_up_new_snapshots():
    n = 4096
    sim, opp, ro, snaps = _graphed(n, 1, 30)
    assert ro.graph is not None
    red, eager, _ = _replay_and_eager(sim, opp, ro)
    assert torch.allclose(red, eager, rtol=0, atol=1e-5)
    other, other_rms = _snapshot(77)
    opp.set(0, other, other_rms)
    red2, eager2, before = _replay_and_eager(sim, opp, ro)
    assert torch.allclose(red2, eager2, rtol=0, atol=1e-5)
    # the new snapshot, not the old one, played this replay
    old = Opponent(n, slots=1, device=DEV, policy_dtype=torch.bfloat16, deterministic=True)
    old.set(0, *snaps[0])
    shadow = SimpleNamespace(obs=before, actions=torch.zeros_like(sim.actions))
    old.act(shadow)
    assert (shadow.actions[:, 2:] - red2).abs().max() > 1e-2
    assert torch.isfinite(ro.buf.values).all()


def test_graphed_rollout_with_four_slots_plays_each_slice_with_its_own_snapshot():
    n, K = 4096, 4
    sim, opp, ro, snaps = _graphed(n, K, 40)
    red, eager, before = _replay_and_eager(sim, opp, ro)
    assert torch.allclose(red, eager, rtol=0, atol=1e-5)
    for k in range(K):
        b0, b1 = opp.slot_range(k)
        errs = []
        for a, r in snaps:  # every snapshot's fp32 answer on this slice: slot k's own is the only close one
            inv = 1.0 / (r.std.float() + 1e-8)
            with torch.no_grad():
                x = torch.clamp(torch.addcmul(-r.mean.float() * inv, mirror_frames(before[b0:b1, 2:].reshape(-1, 66)), inv), -10, 10)
                want = mirror_actions(a.actor_mean(x).view(-1, 2, 3))
            errs.append(float((red[b0:b1] - want).abs().max()))
        assert errs[k] < 5e-2 and all(e > 3 * errs[k] for j, e in enumerate(errs) if j != k), (k, errs)


def _host_match(sim, agent, rms, opp, steps):
    """The match of evaluate_match (deterministic blue) from the sim's current states, counted on the host from
    sim.score at every done: (n, 5) wins, draws, losses, goals for, goals against per env."""
    n = sim.num_envs
    inv = 1.0 / (rms.std.float() + 1e-8)
    shift = -rms.mean.float() * inv
    host = np.zeros((n, 5), np.int64)
    for _ in range(steps):
        with torch.no_grad():
            x = torch.clamp(torch.addcmul(shift, sim.obs[:, :2].reshape(-1, 66), inv), -10.0, 10.0)
            sim.actions[:, :2] = agent.actor_mean(x).view(n, 2, 3)
        opp.act(sim)
        sim.step(sim.actions, auto_reset=True)
        done, score = sim.done.cpu().numpy().astype(bool), sim.score.cpu().numpy().astype(np.int64)
        diff = score[:, 0] - score[:, 1]
        host[done] += np.stack([diff > 0, diff == 0, diff < 0, score[:, 0], score[:, 1]], 1)[done]
    return host


@pytest.mark.parametrize("start", ["reset", "goal_mouth_states"])
def test_evaluate_match_counts_against_a_host_loop(start):
    """evaluate_match on 512 envs, 4 slots, max_steps 50, two episodes: per slot wins + draws + losses = the episodes,
    the counts equal a host loop over sim.score at done, and goals for / against add up to the statistics' goals.
    'reset': evaluate_match resets the envs itself (seeded).  'goal_mouth_states': it plays from installed states at
    step 0 whose ball is about to cross a goal line (reset=False), so that the match has goals for certain."""
    n, K, episodes = 512, 4, 2
    cfg = dict(P.CONFIG)
    cfg["simulation"] = {"max_steps": 50}
    sim = BatchedSoccerSim(n, config=cfg, device=DEV, seed=5)
    agent, rms = _snapshot(50)
    opp = Opponent(n, slots=K, device=DEV, deterministic=True)
    for k in range(K):
        opp.set(k, *_snapshot(60 + k))
    if start == "goal_mouth_states":
        rng = np.random.default_rng(8)
        states = [dict(P.random_state(rng, "goal"), steps=0, score=(0, 0)) for _ in range(n)]
        recs = np.frombuffer(b"".join(bytes(P.oracle_to_dev_state(s)) for s in states), np.uint8)
        sim.load_states(None, torch.from_numpy(recs.reshape(n, _capi.ENV_STATE_BYTES).copy()))
        sim.obs.copy_(torch.from_numpy(np.stack([s["obs"] for s in states])).to(DEV))
    sim.stats(reset=True)
    snap = sim.state_dict()
    if start == "reset":
        res = evaluate_match(sim, agent, rms, opp, episodes=episodes, seed=123)
    else:
        res = evaluate_match(sim, agent, rms, opp, episodes=episodes, reset=False)
    st = sim.stats()
    assert [r["slot"] for r in res] == list(range(K))
    for r in res:
        assert r["wins"] + r["draws"] + r["losses"] == r["episodes"] == episodes * r["envs"]
    assert sum(r["goals_for"] for r in res) == st["goals_blue"] and sum(r["goals_against"] for r in res) == st["goals_red"]
    if start == "goal_mouth_states":
        assert st["goals_blue"] > 0 and st["goals_red"] > 0 and sum(r["wins"] + r["losses"] for r in res) > 0, st
    # the same match, counted on the host
    sim.load_state_dict(snap)
    if start == "reset":
        sim.reset(_capi.MODE_FULL_RANDOM, seed=123)
    host = _host_match(sim, agent, rms, opp, episodes * 50)
    for k, r in enumerate(res):
        b0, b1 = opp.slot_range(k)
        want = dict(zip(("wins", "draws", "losses", "goals_for", "goals_against"), host[b0:b1].sum(0).tolist()))
        assert {key: r[key] for key in want} == want, (k, r, want)
