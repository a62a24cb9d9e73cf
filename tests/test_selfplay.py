"""Self-play against frozen snapshots (marl_soccer_b200/selfplay.py), without a GPU: the mirror convention feature by
feature and against the oracle (observations and one step of the physics), the fp32 Opponent, the actor-only
PackedPolicy, and the argument checks of msoc_team_inputs."""
import ctypes as C
import math
from types import SimpleNamespace

import numpy as np
import pytest
import torch

import oracle_lib as O
import parity_util as P
from selfplay_util import mirror_obs, mirror_state
from marl_soccer_b200 import _capi, build
from marl_soccer_b200.rollout import Agent, PackedPolicy, RunningMeanStd
from marl_soccer_b200.selfplay import NEGATED, Opponent, mirror_actions, mirror_frames


def _frames(rng, shape):
    x = rng.normal(0, 2, shape).astype(np.float32)
    f = x.reshape(*shape[:-1], -1, 22)
    f[..., 2] = rng.uniform(-1, 1, f.shape[:-1]).astype(np.float32)
    flat = f.reshape(-1, 22)
    if flat.shape[0] >= 5:  # the angle's edge cases, and a frame of negative zeros
        flat[:4, 2] = [0.0, -0.0, 1.0, -1.0]
        flat[4, :] = -0.0
    return x


def test_mirror_follows_the_table_feature_by_feature_in_torch_and_numpy():
    rng = np.random.default_rng(0)
    for shape in ((22,), (7, 66), (3, 5, 22), (2, 4, 66)):
        x = _frames(rng, shape)
        m_np = mirror_frames(x)
        m_t = mirror_frames(torch.from_numpy(x))
        assert m_np.dtype == np.float32 and m_np.shape == x.shape and m_t.shape == x.shape
        assert m_np.tobytes() == m_t.numpy().tobytes()  # bit for bit
        f, g = x.reshape(-1, 22), m_np.reshape(-1, 22)
        for j in range(22):
            if j == 2:
                want = np.where(f[:, 2] >= 0, np.float32(1) - f[:, 2], np.float32(-1) - f[:, 2]).astype(np.float32)
            elif j in NEGATED:
                want = -f[:, j]
            else:
                want = f[:, j]
            assert want.tobytes() == g[:, j].tobytes(), j
    # both zeros map to 1; +-1 map to the zeros of the other sign's branch
    a = np.array([0.0, -0.0, 1.0, -1.0, 0.25, -0.25], np.float32)
    x = np.zeros((6, 22), np.float32)
    x[:, 2] = a
    assert mirror_frames(x)[:, 2].tolist() == [1.0, 1.0, 0.0, 0.0, 0.75, -0.75]
    assert mirror_frames(x)[2, 2] == 0.0 and not np.signbit(mirror_frames(x)[2, 2])
    x = torch.from_numpy(x)
    assert mirror_frames(x)[:, 2].tolist() == [1.0, 1.0, 0.0, 0.0, 0.75, -0.75]
    assert torch.equal(x[:, 2], torch.from_numpy(a))  # the input is not modified
    with pytest.raises(ValueError):
        mirror_frames(np.zeros((3, 21), np.float32))


def test_mirror_actions():
    a = np.array([[0.5, -0.25, 1.0], [-1.0, 0.0, -0.75]], np.float32)
    assert mirror_actions(a).tolist() == [[0.5, 0.25, -1.0], [-1.0, -0.0, 0.75]]
    assert torch.equal(mirror_actions(torch.from_numpy(a)), torch.from_numpy(mirror_actions(a)))
    assert np.array_equal(mirror_actions(mirror_actions(a)), a) and a[0, 1] == -0.25
    with pytest.raises(ValueError):
        mirror_actions(np.zeros((2, 4)))


def _mirror_case_states(n, seed):
    rng = np.random.default_rng(seed)
    kinds = ("open", "walls", "goal")
    return [P.random_state(rng, kinds[i % 3]) for i in range(n)]


def _angle_aware_err(a, b):
    """max |a - b| over rows of 22-float frames; the angle feature is compared modulo 2 (+1 and -1 are the same angle)."""
    a = np.asarray(a, np.float64).reshape(-1, 22).copy()
    b = np.asarray(b, np.float64).reshape(-1, 22).copy()
    da = np.abs(P.wrap((a[..., 2] - b[..., 2]) * math.pi)) / math.pi
    a[..., 2] = b[..., 2] = 0.0
    return float(max(np.abs(a - b).max(), da.max()))


def test_mirrored_red_view_is_the_blue_view_of_the_mirrored_state_on_the_oracle():
    """512 states (open, walls, goal) and their mirror images: the oracle's observation rows (the stacked history and the
    frames of the current pose) of red in S, mirrored, are blue's rows in M(S), and the other way round."""
    worst = 0.0
    for s in _mirror_case_states(512, 11):
        m = mirror_state(s)
        for a_obs, b_obs in ((s["obs"], m["obs"]),
                             (P.frames_of_pose(P.pose_of(s)), P.frames_of_pose(P.pose_of(m)))):
            a_obs, b_obs = np.asarray(a_obs, np.float32), np.asarray(b_obs, np.float32)
            worst = max(worst, _angle_aware_err(mirror_frames(a_obs[2:]), b_obs[:2]),
                        _angle_aware_err(mirror_frames(a_obs[:2]), b_obs[2:]))
    P.record("selfplay_mirror_obs_oracle", {"states": 512, "worst_abs_error": worst})
    assert worst < 1e-4, worst


def test_one_oracle_step_commutes_with_the_mirror():
    """step(S; blue b, red r) mirrored = step(M(S); blue mirror(r), red mirror(b)) within the parity bands (DESIGN.md
    section 3) for every env without a contact on either side; goal flags negated, scores swapped, done equal.  An env
    where a goal falls is compared on those alone: the soft reset after a goal draws the new positions from the env's
    own spawn stream, and those of M(S) are not the mirror images of those of S."""
    n = 512
    states = _mirror_case_states(n, 12)
    mirrored = [mirror_state(s) for s in states]
    rng = np.random.default_rng(13)
    act = rng.uniform(-1.2, 1.2, (n, 4, 3)).astype(np.float32)
    act_m = np.concatenate([mirror_actions(act[:, 2:]), mirror_actions(act[:, :2])], axis=1)
    ora, ora_m = O.OracleVec(n, P.CONFIG, seed=0), O.OracleVec(n, P.CONFIG, seed=0)
    ora.set_states(states)
    ora_m.set_states(mirrored)
    o, _, d, g = ora.step(act, auto_reset=False)
    o_m, _, d_m, g_m = ora_m.step(act_m, auto_reset=False)
    edge = P.goal_knife_edge(states) | P.goal_knife_edge(mirrored)
    assert np.array_equal(d, d_m)
    assert np.array_equal(g[~edge], -g_m[~edge])
    compared, goals, worst = 0, int(np.abs(g).sum()), {}
    for i in range(n):
        e, e_m = ora.env(i), ora_m.env(i)
        s1, s1_m = e.get_state(), e_m.get_state()
        assert s1["score"] == s1_m["score"][::-1] and s1["steps"] == s1_m["steps"]
        if edge[i] or g[i] or e.contact_count() or e_m.contact_count():
            continue
        c = P.compare_state(mirror_state(dict(s1, cache=[], obs=None)), s1_m)
        c["obs"] = P.compare_obs(mirror_obs(o[i]), o_m[i])
        for k, v in c.items():
            worst[k] = max(worst.get(k, 0.0), v)
        compared += 1
    P.record("selfplay_mirror_step_oracle", {"envs": n, "contact_free_compared": compared, "goals": goals,
                                             "worst_violation_ratio": {k: round(v, 3) for k, v in worst.items()}})
    assert compared >= n // 4 and goals > 0, (compared, goals)
    assert max(worst.values()) <= 1.0, worst


def _agents(k, seed):
    torch.manual_seed(seed)
    out = []
    for j in range(k):
        a = Agent()
        with torch.no_grad():
            for p in a.parameters():
                p.add_(0.3 * torch.randn_like(p))  # outputs of order one, so that the slots differ visibly
        r = RunningMeanStd((66,), "cpu")
        r.mean = torch.randn(66, dtype=torch.float64) * 0.2
        r.var = torch.rand(66, dtype=torch.float64) + 0.5
        out.append((a, r))
    return out


def _expected_red(agent, rms, obs_rows):
    """(m, 2, 66) red rows -> red actions (m, 2, 3) of a snapshot playing its mean (the formula of Opponent.act)."""
    inv = 1.0 / (rms.std.float() + 1e-8)
    x = torch.clamp(torch.addcmul(-rms.mean.float() * inv, mirror_frames(obs_rows.reshape(-1, 66)), inv), -10.0, 10.0)
    with torch.no_grad():
        return mirror_actions(agent.actor_mean(x).view(-1, 2, 3))


def test_fp32_opponent_plays_each_slice_with_its_own_snapshot():
    n, K = 11, 3
    snaps = _agents(K, 5)
    opp = Opponent(n, slots=K, device="cpu", deterministic=True)
    params = [p.data_ptr() for p in opp.agents[0].parameters()]
    for k, (a, r) in enumerate(snaps):
        opp.set(k, a, r)
    assert [p.data_ptr() for p in opp.agents[0].parameters()] == params  # copied in place
    assert [opp.slot_range(k) for k in range(K)] == [(0, 3), (3, 7), (7, 11)]
    g = torch.Generator().manual_seed(1)
    sim = SimpleNamespace(obs=torch.randn((n, 4, 66), generator=g), actions=torch.randn((n, 4, 3), generator=g))
    obs0, blue0 = sim.obs.clone(), sim.actions[:, :2].clone()
    opp.act(sim)
    assert torch.equal(sim.obs, obs0) and torch.equal(sim.actions[:, :2], blue0)
    for k, (a, r) in enumerate(snaps):
        b0, b1 = opp.slot_range(k)
        want = _expected_red(a, r, obs0[b0:b1, 2:])
        assert torch.allclose(sim.actions[b0:b1, 2:], want, atol=1e-6), k
        other = _expected_red(*snaps[(k + 1) % K], obs0[b0:b1, 2:])
        assert (sim.actions[b0:b1, 2:] - other).abs().max() > 1e-2, k
    # sampling: the snapshot's actor_logstd; a tiny std gives the mean back, std 1 does not
    sto = Opponent(n, slots=1, device="cpu")
    a, r = snaps[0]
    with torch.no_grad():
        a.actor_logstd.fill_(-30.0)
    sto.set(0, a, r)
    sto.act(sim)
    assert torch.allclose(sim.actions[:, 2:], _expected_red(a, r, obs0[:, 2:]), atol=1e-6)
    with torch.no_grad():
        a.actor_logstd.fill_(0.0)
    sto.set(0, a, r)
    sto.act(sim)
    assert (sim.actions[:, 2:] - _expected_red(a, r, obs0[:, 2:])).abs().max() > 0.1


def test_opponent_rejects_bad_arguments():
    with pytest.raises(ValueError):
        Opponent(0)
    with pytest.raises(ValueError):
        Opponent(4, slots=0, device="cpu")
    with pytest.raises(ValueError):
        Opponent(4, device="cpu", policy_dtype=torch.float16)
    with pytest.raises(ValueError):
        Opponent(4, device="cpu", policy_dtype=torch.bfloat16)
    opp = Opponent(4, slots=2, device="cpu")
    with pytest.raises(IndexError):
        opp.set(2, Agent(), RunningMeanStd((66,), "cpu"))
    with pytest.raises(ValueError):
        opp.act(SimpleNamespace(obs=torch.zeros((5, 4, 66)), actions=torch.zeros((5, 4, 3))))


def test_actor_only_packed_policy_is_the_actor():
    """PackedPolicy(critic=False): the same packing with a stack of one net computes agent.actor_mean and the
    log-probabilities, returns no value, and follows refresh()."""
    torch.manual_seed(3)
    a = Agent()
    with torch.no_grad():
        for p in a.parameters():
            p.add_(0.05 * torch.randn_like(p))
    pp = PackedPolicy(a, torch.float32, critic=False)
    assert pp.w0.shape == (520, 72) and all(w.shape[0] == 1 for w in pp.w)
    x = torch.randn(41, 66)
    x72 = torch.zeros(41, PackedPolicy.IN)
    x72[:, :66] = x
    mean, value = pp(x72)
    assert value is None and torch.allclose(mean, a.actor_mean(x), atol=1e-5)
    full_mean, _ = PackedPolicy(a, torch.float32)(x72)
    assert torch.allclose(mean, full_mean, atol=1e-6)
    action, logprob, value = pp.act(x72)
    _, ref_logprob, _, _ = a.get_action_and_value(x, action)
    assert value is None and torch.allclose(logprob, ref_logprob, atol=1e-4)
    with torch.no_grad():
        a.actor_mean[0].weight.mul_(2.0)
    pp.refresh()
    assert torch.allclose(pp(x72)[0], a.actor_mean(x), atol=1e-5)


def test_team_inputs_rejects_bad_arguments_without_a_device():
    L = C.CDLL(build.build())
    _capi.declare(L)
    buf = (C.c_float * 64)()
    p = C.c_void_p(C.addressof(buf))
    assert L.msoc_team_inputs(p, 1, 2, p, p, p, None, None, None) == -1
    assert b"team" in L.msoc_last_error()
    assert L.msoc_team_inputs(p, 1, -1, p, p, p, None, None, None) == -1
    for team in (0, 1):
        assert L.msoc_team_inputs(None, 1, team, p, p, p, None, None, None) == -1
        assert L.msoc_team_inputs(p, 1, team, None, p, p, None, None, None) == -1
        assert L.msoc_team_inputs(p, 1, team, p, None, p, None, None, None) == -1
        assert L.msoc_team_inputs(p, 1, team, p, p, None, None, None, None) == -1
        assert L.msoc_team_inputs(p, 0, team, p, p, p, None, None, None) == -1
        assert L.msoc_team_inputs(p, -3, team, p, p, p, None, None, None) == -1
        assert b"msoc_team_inputs" in L.msoc_last_error()
    assert "msoc_team_inputs" in _capi.EXPORTS
