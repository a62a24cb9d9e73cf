"""Pins of the CPU oracle (oracle/soccer_oracle.c).  The reference's arithmetic lives in pymunk, which is
absent here (parity unpinned at that boundary, SURVEY.md section 8c); what CAN be pinned is checked:
Random123 known-answer vectors of the Philox spawn stream, the observation layout constants of the
reference's test_rewards.py:37-58, the reference's spawn boxes (game/game.py:129-249), and closed-form
answers of the restated step for contact-free motion and single contacts (SURVEY.md appendices A, B)."""
import math

import numpy as np
import pytest

import oracle_lib as O

CFG = O.DEFAULT_CONFIG
DT = 1.0 / 60.0


def test_reference_config_matches_restated_defaults():
    assert O.load_reference_config() == CFG


def test_philox_known_answers():
    # Random123 kat_vectors: philox4x32_10
    assert O.philox([0, 0, 0, 0], [0, 0]) == [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]
    assert O.philox([0xFFFFFFFF] * 4, [0xFFFFFFFF] * 2) == [0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD]
    assert O.philox([0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344], [0xA4093822, 0x299F31D0]) == [
        0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1]


def blank_state(**kw):
    s = {"pos": np.array([[200.0, 198.0], [200.0, 396.0], [600.0, 198.0], [600.0, 396.0], [400.0, 300.0]]),
         "vel": np.zeros((5, 2)), "ang": np.array([0.0, 0.0, math.pi, math.pi, 0.0]), "angvel": np.zeros(5),
         "vbias": np.zeros((5, 2)), "wbias": np.zeros(5), "steps": 0, "score": (0, 0), "mode": 1,
         "spawn_count": 0, "seed": 0, "obs": np.zeros((4, 66), np.float32), "cache": []}
    s.update(kw)
    return s


def test_fixed_spawn_and_observation_layout():
    """test_rewards.py:37-58: FRAME 22 x STACK 3, newest frame last; slots 4 teammate, 7/10 opponents,
    13 ball, 16 own goal, 19 opponent goal; magnitudes are / hypot(800, 600) = 1000."""
    e = O.OracleEnv(seed=1)
    obs = e.reset(O.MODE_FIXED)
    st = e.get_state()
    assert np.allclose(st["pos"], [[200, 198], [200, 396], [600, 198], [600, 396], [400, 300]])
    assert obs.shape == (4, 66) and obs.dtype == np.float32
    f = obs.reshape(4, 3, 22)
    assert np.array_equal(f[:, 0], f[:, 1]) and np.array_equal(f[:, 1], f[:, 2])  # 3 copies after reset
    a0 = f[0, 2]
    assert np.allclose(a0[0:4], 0.0)                                   # v, angle 0, w
    assert np.allclose(a0[4:7], [0.0, 1.0, 0.198], atol=1e-6)           # teammate (agent_1) straight up, 198 px
    d2 = math.hypot(400, 0); assert np.allclose(a0[7:10], [1.0, 0.0, d2 / 1000], atol=1e-6)  # opp1 = agent_2
    d3 = math.hypot(400, 198); assert np.allclose(a0[10:13], [400 / d3, 198 / d3, d3 / 1000], atol=1e-6)
    db = math.hypot(200, 102); assert np.allclose(a0[13:16], [200 / db, 102 / db, db / 1000], atol=1e-6)
    dg = math.hypot(190, 102); assert np.allclose(a0[16:19], [-190 / dg, 102 / dg, dg / 1000], atol=1e-6)  # own goal (10,300)
    do = math.hypot(590, 102); assert np.allclose(a0[19:22], [590 / do, 102 / do, do / 1000], atol=1e-6)   # red goal (790,300)
    a2 = f[2, 2]
    assert abs(abs(a2[2]) - 1.0) < 1e-6                                # red faces pi -> +-1
    assert np.allclose(a2[4:7], [0.0, 1.0, 0.198], atol=1e-6)           # teammate of agent_2 is agent_3
    assert np.allclose(a2[7:10], [-1.0, 0.0, 0.4], atol=1e-6)           # red sees blue (0, 1) in index order
    assert a2[16] > 0 and a2[19] < 0                                    # own goal right, opponent goal left


def test_spawn_boxes_of_the_three_modes():
    n = 4000
    v = O.OracleVec(n, CFG, seed=11)
    v.reset(O.MODE_RANDOM, seed=3)
    p = np.array([s["pos"] for s in v.get_states()])
    assert (p[:, :2, 0] >= 30).all() and (p[:, :2, 0] < 380).all()      # blue left half
    assert (p[:, 2:4, 0] >= 420).all() and (p[:, 2:4, 0] < 770).all()   # red right half
    assert (p[:, :4, 1] >= 30).all() and (p[:, :4, 1] < 570).all()
    assert (np.abs(p[:, 4] - [400, 300]) <= 40).all()                   # ball around the centre
    v.reset(O.MODE_FULL_RANDOM, seed=4)
    p = np.array([s["pos"] for s in v.get_states()])
    cx = np.minimum(np.abs(p[:, 0, 0] - 18), np.abs(p[:, 0, 0] - 782)) <= 5.0
    cy = np.minimum(np.abs(p[:, 0, 1] - 18), np.abs(p[:, 0, 1] - 582)) <= 5.0
    frac = np.mean(cx & cy)
    assert 0.72 < frac < 0.79                                           # 75 % corner spawns (+ a few by chance)
    assert (p[:, 2:, 0] >= 30).all() and (p[:, 2:, 0] < 770).all()
    # seeds: env i is seeded with seed + global index; same seed -> same spawn, other seed -> different
    a = v.reset(O.MODE_FULL_RANDOM, seed=9).copy()
    b = v.reset(O.MODE_FULL_RANDOM, seed=9)
    assert np.array_equal(a, b) and not np.array_equal(a, v.reset(O.MODE_FULL_RANDOM, seed=10))


def test_contact_free_step_closed_form():
    """SURVEY.md appendix B: p += v dt (old v); v = (v + R(a) F / m dt) * 0.99, clamp 200; w = (w + T/I dt) * 0.99."""
    e = O.OracleEnv(seed=0)
    s = blank_state(vel=np.array([[10.0, -5.0], [0, 0], [3.0, 4.0], [0, 0], [30.0, 40.0]]),
                    ang=np.array([0.5, 0.0, math.pi, 2.0, 0.0]), angvel=np.array([1.0, 0, -2.0, 0, 3.0]))
    e.set_state(s)
    act = np.array([[0.01, 0.02, 0.5], [0, 0, 0], [1.5, -0.3, -1.0], [0, 0, 0]], np.float32)
    obs, rew, done, goal = e.step(act)
    st = e.get_state()
    for i, (a, u) in enumerate(zip(s["ang"][:4], act)):
        u = np.clip(u, -1, 1)
        F = np.array([np.float32(u[0]) * np.float32(150000.0), np.float32(u[1]) * np.float32(150000.0)], np.float64)
        Fw = np.array([F[0] * math.cos(a) - F[1] * math.sin(a), F[0] * math.sin(a) + F[1] * math.cos(a)])
        v = (s["vel"][i] + Fw / 10.0 * DT) * 0.99
        if np.linalg.norm(v) > 200:
            v = v / np.linalg.norm(v) * 200
        assert np.allclose(st["pos"][i], s["pos"][i] + s["vel"][i] * DT, atol=1e-12)
        assert np.allclose(st["vel"][i], v, atol=1e-9)
        w = (s["angvel"][i] + float(np.float32(u[2]) * np.float32(1000.0)) / 100.0 * DT) * 0.99
        assert abs(st["angvel"][i] - w) < 1e-12 and abs(st["ang"][i] - (a + s["angvel"][i] * DT)) < 1e-12
    assert np.allclose(st["vel"][4], s["vel"][4] * 0.97) and st["angvel"][4] == 3.0  # ball: no angular damping
    # reward = 0.002 * sum(d_prev - d) + 0.1 * (D_prev - D) - 1e-5 (game/game.py:324-375)
    bp0, bp1 = s["pos"][4], st["pos"][4]
    prox = sum(np.linalg.norm(s["pos"][i] - bp0) - np.linalg.norm(st["pos"][i] - bp1) for i in (0, 1))
    move = np.linalg.norm(bp0 - [790, 300]) - np.linalg.norm(bp1 - [790, 300])
    assert abs(rew[0] - (0.002 * prox + 0.1 * move - 1e-5)) < 1e-12 and rew[0] == rew[1]
    assert not done and goal == 0 and st["steps"] == 1


def test_ball_wall_bounce_restitution():
    """Single circle-segment contact: post-step normal velocity = -e * (pre-step normal velocity), e = 0.95^2."""
    e = O.OracleEnv(seed=0)
    s = blank_state(pos=np.array([[200.0, 198.0], [200.0, 396.0], [600.0, 198.0], [600.0, 396.0], [400.0, 23.0]]),
                    vel=np.array([[0, 0], [0, 0], [0, 0], [0, 0], [30.0, -120.0]]))
    e.set_state(s)
    e.step(np.zeros((4, 3), np.float32))
    st = e.get_state()
    assert e.contact_count() == 1
    assert abs(st["vel"][4][1] - 0.9025 * 120.0) < 1e-9
    assert 0.0 < st["vel"][4][0] < 30.0 * 0.97 + 1e-9      # tangential: friction only slows it
    assert len(st["cache"]) == 1 and st["cache"][0][0] == 42 and st["cache"][0][2] == 0  # ball x bottom wall, age 0


def test_goal_soft_reset_and_truncation():
    cfg = {**CFG, "rewards": {**CFG["rewards"], "score_difference_multiplier": 5.0}, "simulation": {"max_steps": 3}}
    e = O.OracleEnv(cfg, seed=2)
    e.reset(O.MODE_FIXED)
    s = e.get_state()
    s["pos"][4] = [788.0, 300.0]; s["vel"][4] = [200.0, 0.0]; s["angvel"][4] = 2.5
    e.set_state(s)
    obs, rew, done, goal = e.step(np.zeros((4, 3), np.float32))
    st = e.get_state()
    assert goal == 1 and st["score"] == (1, 0) and not done
    b0, b1 = np.array([788.0, 300.0]), np.array([788.0 + 200.0 / 60.0, 300.0])
    prox = sum(np.linalg.norm(s["pos"][i] - b0) - np.linalg.norm(s["pos"][i] - b1) for i in (0, 1))
    move = np.linalg.norm(b0 - [790, 300]) - np.linalg.norm(b1 - [790, 300])
    assert abs(rew[0] - (0.002 * prox + 0.1 * move + 4.0 - 1e-5)) < 1e-9  # goal reward on top of the shaping
    assert np.allclose(st["pos"][4], [400, 300]) and np.allclose(st["vel"], 0) and st["angvel"][4] == 2.5  # soft reset
    e.step(np.zeros((4, 3), np.float32))
    obs, rew, done, goal = e.step(np.zeros((4, 3), np.float32))
    assert done and rew == (5.0, 5.0)        # terminal step: reward REPLACED by multiplier * (blue - red)
    obs, rew, done, goal = e.step(np.zeros((4, 3), np.float32))
    assert done                              # stepping after done is allowed (test_rewards.py:485-490)


def test_arbiter_cache_persistence_three_steps():
    """An arbiter survives collision_persistence = 3 steps without contact, then is dropped."""
    e = O.OracleEnv(seed=0)
    s = blank_state(pos=np.array([[200.0, 198.0], [200.0, 396.0], [600.0, 198.0], [600.0, 396.0], [400.0, 23.0]]),
                    vel=np.array([[0, 0], [0, 0], [0, 0], [0, 0], [0.0, -120.0]]))
    e.set_state(s)
    ages = []
    for _ in range(5):
        e.step(np.zeros((4, 3), np.float32))
        ages.append([c[2] for c in e.get_state()["cache"]])
    assert ages == [[0], [1], [2], [], []]
