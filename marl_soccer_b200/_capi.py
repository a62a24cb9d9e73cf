"""ctypes binding of the C-ABI in include/msoc.h (marl_soccer_b200/libmsoc.so).

The library holds the hand-written sm_100a kernels; there is NO CPU fallback: if the shared
library is missing or no CUDA device is present the calls raise.  Struct layouts mirror
include/msoc.h field by field.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MSOC_LIB", os.path.join(PKG_DIR, "libmsoc.so"))  # MSOC_LIB: kernel A/B experiments

N_AGENTS, ACT_DIM, FRAME, STACK, OBS, MAX_CACHE = 4, 3, 22, 3, 66, 32
MODE_RANDOM, MODE_FIXED, MODE_FULL_RANDOM = 0, 1, 2
STEP_AUTO_RESET = 1
STEP_GENERAL_PATH = 2  # debugging / tests: no light / pair / multi class

# every symbol include/msoc.h declares (tests check that the library exports all of them)
EXPORTS = (
    "msoc_last_error", "msoc_version", "msoc_create", "msoc_destroy", "msoc_num_envs", "msoc_reset",
    "msoc_step", "msoc_step_host", "msoc_reset_host", "msoc_read_counters", "msoc_get_state",
    "msoc_set_state", "msoc_get_obs_host", "msoc_step_host_frames", "msoc_stats_device", "msoc_stats_read",
    "msoc_launch_count", "msoc_device_buffers", "msoc_debug_errors", "msoc_last_class_counts", "msoc_policy_inputs",
    "msoc_render", "msoc_render_host", "msoc_save_states", "msoc_load_states", "msoc_team_inputs",
    "msoc_step_teams",
)


class MsocConfig(C.Structure):
    _fields_ = [(k, C.c_float) for k in (
        "max_velocity", "agent_mass", "ball_mass", "agent_moment", "ball_moment", "agent_friction",
        "ball_friction", "action_force_max", "action_torque_max", "max_angular_velocity",
        "ball_proximity_multiplier", "move_ball_to_goal_multiplier", "goal_scored_reward",
        "goal_conceded_penalty", "alive_penalty", "score_difference_multiplier")] + [
        ("max_steps", C.c_int32), ("reserved", C.c_int32)]


class MsocEnvState(C.Structure):
    _fields_ = [
        ("pos", C.c_float * 2 * 5), ("vel", C.c_float * 2 * 5), ("ang", C.c_float * 4),
        ("angvel", C.c_float * 5), ("vbias", C.c_float * 2 * 5), ("wbias", C.c_float * 4),
        ("ep_return", C.c_float), ("steps", C.c_int32), ("score", C.c_int32 * 2), ("mode", C.c_int32),
        ("spawn_count", C.c_uint32), ("cache_count", C.c_uint32), ("seed", C.c_uint64),
        ("cache_info", C.c_uint32 * MAX_CACHE), ("cache_jn", C.c_float * MAX_CACHE),
        ("cache_jt", C.c_float * MAX_CACHE),
        # observation history as poses (include/msoc.h): [0] behind frame t-2, [1] behind frame t-1
        ("hist_valid", C.c_uint32), ("reserved0", C.c_uint32),
        ("hist_pos", C.c_float * 2 * 5 * 2), ("hist_vel", C.c_float * 2 * 4 * 2),
        ("hist_ang", C.c_float * 4 * 2), ("hist_angvel", C.c_float * 4 * 2),
    ]


ENV_STATE_BYTES = 808
assert C.sizeof(MsocEnvState) == ENV_STATE_BYTES
# the same record as a NumPy structured dtype (offsets from the ctypes struct): a host snapshot is an array of these
ENV_STATE_DTYPE = np.dtype(MsocEnvState)


def _field_layout():
    """name -> (byte offset, shape, torch dtype) of every msoc_env_state field."""
    import torch
    scalars = {C.c_float: torch.float32, C.c_int32: torch.int32, C.c_uint32: torch.uint32, C.c_uint64: torch.uint64}
    out = {}
    for name, ctype in MsocEnvState._fields_:
        shape = []
        while hasattr(ctype, "_length_"):  # c_float * 2 * 5 is an array of 5 arrays of 2
            shape.append(ctype._length_)
            ctype = ctype._type_
        out[name] = (getattr(MsocEnvState, name).offset, tuple(shape), scalars[ctype])
    return out


def state_fields(t) -> dict:
    """Named, writable typed views of a (n, 808) uint8 tensor of msoc_env_state records, on any device: e.g.
    state_fields(t)["pos"] is (n, 5, 2) float32, ["seed"] (n,) uint64, ["cache_info"] (n, 32) uint32.  Writes through
    the views land in `t`.  (torch has few arithmetic kernels for uint32 / uint64; view those as int32 / int64 for
    arithmetic.)"""
    if t.dim() != 2 or t.shape[1] != ENV_STATE_BYTES or t.dtype.itemsize != 1 or t.dtype.is_floating_point:
        raise ValueError(f"expected a (n, {ENV_STATE_BYTES}) uint8 tensor, got {tuple(t.shape)} {t.dtype}")
    if t.stride(1) != 1 or t.stride(0) % 8 != 0 or t.storage_offset() % 8 != 0:
        raise ValueError("state_fields needs rows of 808 contiguous bytes at 8-byte aligned offsets")
    n = t.shape[0]
    views = {}
    for name, (off, shape, dt) in _field_layout().items():
        count = int(np.prod(shape)) if shape else 1
        v = t[:, off:off + count * dt.itemsize].view(dt)
        views[name] = v.view((n, *shape)) if shape else v.view(n)
    return views


class MsocStats(C.Structure):
    _fields_ = [(k, C.c_double) for k in (
        "episodes", "episode_return_sum", "goals_blue", "goals_red", "env_steps", "contacts",
        "contact_overflow", "nonfinite_actions")]


def make_config(config: dict) -> MsocConfig:
    """config.json dict -> POD with the reference's defaults for absent keys
    (soccer_env.py:63-64; game/game.py:27,262-264,330,430; game/entities.py:11,62)."""
    ph, rw, sim = config.get("physics", {}), config.get("rewards", {}), config.get("simulation", {})
    c = MsocConfig()
    c.max_velocity = float(ph["max_velocity"])
    c.agent_mass = float(ph["agent_mass"])
    c.ball_mass = float(ph["ball_mass"])
    c.agent_moment, c.ball_moment = 100.0, 10.0
    c.agent_friction = float(ph["agent_friction"])
    c.ball_friction = float(ph["ball_friction"])
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


class MsocBuffers(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in ("obs", "actions", "reward", "done", "goal", "score", "mask", "stats")]


class MsocError(RuntimeError):
    pass


_lib = None


def declare(L) -> None:
    """argtypes/restypes of every entry point (also used by tests on the host harness)."""
    vp, u64, i64, u32 = C.c_void_p, C.c_uint64, C.c_int64, C.c_uint32
    L.msoc_last_error.restype = C.c_char_p
    L.msoc_version.restype = C.c_int
    L.msoc_launch_count.restype = u64
    L.msoc_debug_errors.restype = C.c_int
    L.msoc_create.argtypes = [C.POINTER(MsocConfig), i64, C.c_int, u64, u64, C.POINTER(vp)]
    L.msoc_destroy.argtypes = [vp]
    L.msoc_num_envs.argtypes = [vp]
    L.msoc_num_envs.restype = i64
    L.msoc_reset.argtypes = [vp, vp, C.c_int, C.c_int, u64, vp, vp]
    L.msoc_step.argtypes = [vp, vp, vp, vp, vp, vp, vp, u32, vp]
    L.msoc_step_teams.argtypes = [vp, vp, vp, vp, vp, vp, vp, u32, vp]
    L.msoc_step_host.argtypes = [vp, vp, vp, vp, vp, vp, vp, u32, vp]
    L.msoc_step_host_frames.argtypes = [vp, vp, vp, vp, vp, vp, vp, u32, vp]
    L.msoc_reset_host.argtypes = [vp, vp, C.c_int, C.c_int, u64, vp, vp]
    L.msoc_read_counters.argtypes = [vp, vp, vp, vp]
    L.msoc_get_state.argtypes = [vp, vp, i64, vp]
    L.msoc_set_state.argtypes = [vp, vp, i64, vp]
    L.msoc_get_obs_host.argtypes = [vp, vp, i64, vp]
    L.msoc_device_buffers.argtypes = [vp, C.POINTER(MsocBuffers)]
    L.msoc_stats_device.argtypes = [vp, vp, C.c_int, vp]
    L.msoc_stats_read.argtypes = [vp, C.POINTER(MsocStats), C.c_int, vp]
    L.msoc_last_class_counts.argtypes = [vp, C.POINTER(C.c_int32 * 4), vp]
    L.msoc_policy_inputs.argtypes = [vp, i64, vp, vp, vp, vp, vp, vp]
    L.msoc_team_inputs.argtypes = [vp, i64, C.c_int, vp, vp, vp, vp, vp, vp]
    L.msoc_render.argtypes = [vp, vp, i64, C.c_int, C.c_int, vp, vp]
    L.msoc_render_host.argtypes = [vp, vp, i64, C.c_int, C.c_int, vp]
    L.msoc_save_states.argtypes = [vp, vp, i64, vp, vp]
    L.msoc_load_states.argtypes = [vp, vp, i64, vp, vp]


def lib():
    """Load libmsoc.so; raises if it has not been built (python -c 'import __graft_entry__ as g; g.build()')."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise MsocError(
                f"{LIB_PATH} is missing: build the CUDA extension first "
                "(python -m marl_soccer_b200.build).  There is no CPU fallback.")
        L = C.CDLL(LIB_PATH)
        declare(L)
        _lib = L
    return _lib


def check(rc: int) -> None:
    if rc != 0:
        msg = lib().msoc_last_error()
        raise MsocError(f"msoc error {rc}: {msg.decode() if msg else '?'}")
