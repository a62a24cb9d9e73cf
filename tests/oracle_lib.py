"""ctypes binding of the CPU oracle (oracle/liboracle.so).  TEST INFRASTRUCTURE.

Only tests/, __graft_entry__.smoke() and bench.py's CPU-baseline legs import this.
The product package never does.  The oracle restates soccer_simulation/game/game.py,
game/entities.py, soccer_env.py and marl_vecenv.py of the reference plus the Chipmunk2D
step it calls (game/game.py:399); see oracle/soccer_oracle.c for line-level citations.
"""
from __future__ import annotations

import ctypes as C
import json
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
LIB_PATH = os.path.join(ORACLE_DIR, "liboracle.so")

FRAME, OBS, N_PAIRS, MAX_CACHE = 22, 66, 48, 96
MODE_RANDOM, MODE_FIXED, MODE_FULL_RANDOM = 0, 1, 2

# config.json of the reference (soccer_simulation/config.json), restated as the defaults.
DEFAULT_CONFIG = {
    "physics": {"max_velocity": 200, "agent_mass": 10, "ball_mass": 1, "agent_friction": 0.99,
                "ball_friction": 0.97, "action_torque_max": 1000.0},
    "rewards": {"kick_possession_reward": 0.0, "ball_proximity_multiplier": 0.002,
                "move_ball_to_goal_multiplier": 0.1, "alive_penalty": 0.00001,
                "goal_scored_reward": 4.0, "goal_conceded_penalty": 0.0,
                "score_difference_multiplier": 0.0},
    "simulation": {"max_steps": 1000},
}


class OracleConfig(C.Structure):
    _fields_ = [(k, C.c_double) for k in (
        "max_velocity", "agent_mass", "ball_mass", "agent_friction", "ball_friction",
        "agent_moment", "ball_moment", "action_force_max", "action_torque_max", "max_angular_velocity",
        "ball_proximity_multiplier", "move_ball_to_goal_multiplier", "goal_scored_reward",
        "goal_conceded_penalty", "alive_penalty", "score_difference_multiplier")] + [
        ("max_steps", C.c_int32), ("_pad", C.c_int32)]


class OracleState(C.Structure):
    _fields_ = [
        ("pos", C.c_double * 2 * 5), ("vel", C.c_double * 2 * 5), ("ang", C.c_double * 5),
        ("angvel", C.c_double * 5), ("vbias", C.c_double * 2 * 5), ("wbias", C.c_double * 5),
        ("steps", C.c_int32), ("score", C.c_int32 * 2), ("mode", C.c_int32),
        ("spawn_count", C.c_uint32), ("cache_count", C.c_uint32), ("seed", C.c_uint64),
        ("obs", C.c_float * OBS * 4),
        ("cache_pair", C.c_int32 * MAX_CACHE), ("cache_key", C.c_int32 * MAX_CACHE),
        ("cache_age", C.c_int32 * MAX_CACHE),
        ("cache_jn", C.c_double * MAX_CACHE), ("cache_jt", C.c_double * MAX_CACHE),
    ]


def make_config(config: dict | None = None) -> OracleConfig:
    """config.json dict -> POD, with the reference's defaults for absent keys
    (soccer_env.py:63-64, game/game.py:262-264,330,430)."""
    cfg = config if config is not None else DEFAULT_CONFIG
    ph, rw, sim = cfg.get("physics", {}), cfg.get("rewards", {}), cfg.get("simulation", {})
    c = OracleConfig()
    c.max_velocity = float(ph["max_velocity"])
    c.agent_mass = float(ph["agent_mass"])
    c.ball_mass = float(ph["ball_mass"])
    c.agent_friction = float(ph["agent_friction"])
    c.ball_friction = float(ph["ball_friction"])
    c.agent_moment, c.ball_moment = 100.0, 10.0
    c.action_force_max = float(ph.get("action_force_max", 150000.0))
    c.action_torque_max = float(ph.get("action_torque_max", 100000.0))
    c.max_angular_velocity = float(ph.get("max_angular_velocity", ph.get("action_torque_max", 100000.0) / 100.0))
    c.ball_proximity_multiplier = float(rw.get("ball_proximity_multiplier", 0.0))
    c.move_ball_to_goal_multiplier = float(rw["move_ball_to_goal_multiplier"])
    c.goal_scored_reward = float(rw["goal_scored_reward"])
    c.goal_conceded_penalty = float(rw["goal_conceded_penalty"])
    c.alive_penalty = float(rw["alive_penalty"])
    c.score_difference_multiplier = float(rw.get("score_difference_multiplier", 5.0))
    c.max_steps = int(sim["max_steps"])
    return c


_lib = None


def build(force: bool = False) -> str:
    src = os.path.join(ORACLE_DIR, "soccer_oracle.c")
    stale = (not os.path.exists(LIB_PATH)) or (
        os.path.exists(src) and os.path.getmtime(src) > os.path.getmtime(LIB_PATH))
    if force or stale:
        subprocess.run(["make", "-C", ORACLE_DIR, "liboracle.so"], check=True, capture_output=True)
    return LIB_PATH


def lib():
    global _lib
    if _lib is not None:
        return _lib
    build()
    L = C.CDLL(LIB_PATH)
    vp, u64, i64 = C.c_void_p, C.c_uint64, C.c_int64
    fp = np.ctypeslib.ndpointer(np.float32, flags="C_CONTIGUOUS")
    L.oracle_philox4x32_10.argtypes = [C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]
    L.oracle_create.restype = vp
    L.oracle_create.argtypes = [C.POINTER(OracleConfig), u64, u64]
    L.oracle_destroy.argtypes = [vp]
    L.oracle_reset.argtypes = [vp, C.c_int, C.c_int, u64]
    L.oracle_get_obs.argtypes = [vp, fp]
    L.oracle_frames.argtypes = [vp, fp]
    L.oracle_step.argtypes = [vp, fp, vp, C.POINTER(C.c_double), C.POINTER(C.c_uint8), C.POINTER(C.c_int8)]
    L.oracle_get_state.argtypes = [vp, C.POINTER(OracleState)]
    L.oracle_set_state.argtypes = [vp, C.POINTER(OracleState)]
    L.oracle_contact_count.argtypes = [vp]
    L.oracle_contact_count.restype = C.c_int
    L.oracle_vec_create.restype = vp
    L.oracle_vec_create.argtypes = [C.POINTER(OracleConfig), i64, u64, u64]
    L.oracle_vec_destroy.argtypes = [vp]
    L.oracle_vec_env.restype = vp
    L.oracle_vec_env.argtypes = [vp, i64]
    L.oracle_vec_reset.argtypes = [vp, vp, C.c_int, C.c_int, u64, vp]
    L.oracle_vec_step.argtypes = [vp, vp, vp, vp, vp, vp, C.c_int, C.c_int]
    _lib = L
    return L


def philox(ctr, key):
    c = (C.c_uint32 * 4)(*ctr)
    k = (C.c_uint32 * 2)(*key)
    o = (C.c_uint32 * 4)()
    lib().oracle_philox4x32_10(c, k, o)
    return [int(x) for x in o]


# Field order of the flat state dict used by the parity tests (shared with the device wrapper).
STATE_KEYS = ("pos", "vel", "ang", "angvel", "vbias", "wbias", "steps", "score", "mode",
              "spawn_count", "seed", "obs", "cache")


def state_to_dict(S: OracleState) -> dict:
    n = int(S.cache_count)
    return {
        "pos": np.array(S.pos, dtype=np.float64), "vel": np.array(S.vel, dtype=np.float64),
        "ang": np.array(S.ang, dtype=np.float64), "angvel": np.array(S.angvel, dtype=np.float64),
        "vbias": np.array(S.vbias, dtype=np.float64), "wbias": np.array(S.wbias, dtype=np.float64),
        "steps": int(S.steps), "score": (int(S.score[0]), int(S.score[1])), "mode": int(S.mode),
        "spawn_count": int(S.spawn_count), "seed": int(S.seed),
        "obs": np.array(S.obs, dtype=np.float32),
        "cache": [(int(S.cache_pair[k]), int(S.cache_key[k]), int(S.cache_age[k]),
                   float(S.cache_jn[k]), float(S.cache_jt[k])) for k in range(n)],
    }


def dict_to_state(d: dict) -> OracleState:
    S = OracleState()
    for i in range(5):
        for k in range(2):
            S.pos[i][k] = float(d["pos"][i][k])
            S.vel[i][k] = float(d["vel"][i][k])
            S.vbias[i][k] = float(d["vbias"][i][k]) if "vbias" in d else 0.0
        S.ang[i] = float(d["ang"][i]) if i < len(d["ang"]) else 0.0
        S.angvel[i] = float(d["angvel"][i])
        S.wbias[i] = float(d["wbias"][i]) if "wbias" in d else 0.0
    S.steps = int(d.get("steps", 0))
    S.score[0], S.score[1] = (int(x) for x in d.get("score", (0, 0)))
    S.mode = int(d.get("mode", MODE_RANDOM))
    S.spawn_count = int(d.get("spawn_count", 0))
    S.seed = int(d.get("seed", 0))
    obs = d.get("obs")
    if obs is not None:
        obs = np.asarray(obs, dtype=np.float32).reshape(4, OBS)
        for i in range(4):
            for k in range(OBS):
                S.obs[i][k] = float(obs[i, k])
    cache = d.get("cache", [])
    S.cache_count = len(cache)
    for k, (p, key, age, jn, jt) in enumerate(cache):
        S.cache_pair[k], S.cache_key[k], S.cache_age[k] = int(p), int(key), int(age)
        S.cache_jn[k], S.cache_jt[k] = float(jn), float(jt)
    return S


class OracleEnv:
    """One env of the oracle (the Game + the stacking of SoccerEnv)."""

    def __init__(self, config: dict | None = None, seed: int = 0, global_index: int = 0):
        self._L = lib()
        self._cfg = make_config(config)
        self._h = self._L.oracle_create(C.byref(self._cfg), seed, global_index)
        self._owned = True

    @classmethod
    def _borrow(cls, handle):
        self = cls.__new__(cls)
        self._L = lib()
        self._h = handle
        self._owned = False
        return self

    def __del__(self):
        if getattr(self, "_owned", False) and self._h:
            self._L.oracle_destroy(self._h)
            self._h = None

    def reset(self, mode: int = MODE_RANDOM, seed: int | None = None) -> np.ndarray:
        self._L.oracle_reset(self._h, mode, 0 if seed is None else 1, 0 if seed is None else int(seed))
        return self.obs()

    def obs(self) -> np.ndarray:
        o = np.zeros((4, OBS), np.float32)
        self._L.oracle_get_obs(self._h, o)
        return o

    def frames(self) -> np.ndarray:
        """(4, 22): the frames of the current bodies; the 3-frame history is not touched."""
        o = np.zeros((4, FRAME), np.float32)
        self._L.oracle_frames(self._h, o)
        return o

    def step(self, actions):
        a = np.ascontiguousarray(actions, dtype=np.float32).reshape(12)
        o = np.zeros((4, OBS), np.float32)
        r = (C.c_double * 2)()
        d, g = C.c_uint8(), C.c_int8()
        self._L.oracle_step(self._h, a, o.ctypes.data, r, C.byref(d), C.byref(g))
        return o, (r[0], r[1]), bool(d.value), int(g.value)

    def get_state(self) -> dict:
        S = OracleState()
        self._L.oracle_get_state(self._h, C.byref(S))
        return state_to_dict(S)

    def set_state(self, d: dict) -> None:
        S = dict_to_state(d)
        self._L.oracle_set_state(self._h, C.byref(S))

    def contact_count(self) -> int:
        return int(self._L.oracle_contact_count(self._h))


class OracleVec:
    """N envs of the oracle behind the array API of marl_vecenv.SyncMultiAgentVecEnv."""

    def __init__(self, n: int, config: dict | None = None, seed: int = 0, global_offset: int = 0):
        self._L = lib()
        self._cfg = make_config(config)
        self.n = int(n)
        self._h = self._L.oracle_vec_create(C.byref(self._cfg), self.n, seed, global_offset)

    def __del__(self):
        if getattr(self, "_h", None):
            self._L.oracle_vec_destroy(self._h)
            self._h = None

    def env(self, i: int) -> OracleEnv:
        return OracleEnv._borrow(self._L.oracle_vec_env(self._h, i))

    def reset(self, mode: int = MODE_RANDOM, seed: int | None = None, mask=None) -> np.ndarray:
        obs = np.zeros((self.n, 4, OBS), np.float32)
        m = None if mask is None else np.ascontiguousarray(mask, dtype=np.uint8)
        self._L.oracle_vec_reset(self._h, None if m is None else m.ctypes.data, mode,
                                 0 if seed is None else 1, 0 if seed is None else int(seed), obs.ctypes.data)
        return obs

    def step(self, actions, auto_reset: bool = True, nthreads: int = 1, want_obs: bool = True):
        a = np.ascontiguousarray(actions, dtype=np.float32).reshape(self.n, 12)
        obs = np.zeros((self.n, 4, OBS), np.float32) if want_obs else None
        rew = np.zeros((self.n, 2), np.float64)
        done = np.zeros(self.n, np.uint8)
        goal = np.zeros(self.n, np.int8)
        self._L.oracle_vec_step(self._h, a.ctypes.data, None if obs is None else obs.ctypes.data,
                                rew.ctypes.data, done.ctypes.data, goal.ctypes.data,
                                1 if auto_reset else 0, int(nthreads))
        return obs, rew, done, goal

    def get_states(self):
        return [self.env(i).get_state() for i in range(self.n)]

    def set_states(self, states):
        for i, s in enumerate(states):
            self.env(i).set_state(s)


def load_reference_config() -> dict:
    """The shipped copy of the reference's soccer_simulation/config.json (marl_soccer_b200/config.json)."""
    with open(os.path.join(ROOT, "marl_soccer_b200", "config.json")) as f:
        return json.load(f)
