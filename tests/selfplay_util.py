"""Mirror of an oracle state dict about x = 400 (the convention of marl_soccer_b200/selfplay.py and msoc_team_inputs):
agents 0 <-> 2 and 1 <-> 3 swap, the ball stays body 4; x -> 800 - x, vx -> -vx, theta -> wrap(pi - theta), omega ->
-omega (the ball's too), the bias velocities likewise; the score swaps; both history poses are mirrored the same way.
For states with an empty arbiter cache."""
from __future__ import annotations

import math

import numpy as np

import parity_util as P
from marl_soccer_b200.selfplay import mirror_frames

SWAP = [2, 3, 0, 1, 4]


def wrap(a):
    return np.arctan2(np.sin(a), np.cos(a))


def _mirror_pose(d: dict) -> dict:
    pos = np.asarray(d["pos"], np.float64)[SWAP].copy()
    vel = np.asarray(d["vel"], np.float64)[SWAP].copy()
    pos[:, 0] = 800.0 - pos[:, 0]
    vel[:, 0] = -vel[:, 0]
    ang = np.asarray(d["ang"], np.float64)[SWAP].copy()
    ang[:4] = wrap(math.pi - ang[:4])  # the ball's angle plays no part (a circle) and is kept
    angvel = -np.asarray(d["angvel"], np.float64)[SWAP]
    return {"pos": pos, "vel": vel, "ang": ang, "angvel": angvel}


def mirror_state(d: dict, config=None) -> dict:
    assert not d.get("cache"), "mirror_state takes states with an empty cache"
    out = dict(d)
    out.update(_mirror_pose(d))
    vb = np.asarray(d.get("vbias", np.zeros((5, 2))), np.float64)[SWAP].copy()
    vb[:, 0] = -vb[:, 0]
    out["vbias"] = vb
    out["wbias"] = -np.asarray(d.get("wbias", np.zeros(5)), np.float64)[SWAP]
    out["score"] = (d["score"][1], d["score"][0])
    if d.get("hist") is not None:
        out["hist"] = [_mirror_pose(h) for h in d["hist"]]
        out["obs"] = P.obs_of_hist(out["hist"], config)  # what the oracle shows for the mirrored history
    elif d.get("obs") is not None:
        out["obs"] = mirror_obs(d["obs"])
    out["cache"] = []
    return out


def mirror_obs(obs) -> np.ndarray:
    """(..., 4, 66) observation rows of a state -> the rows of its mirrored state (agents swapped, frames mirrored)."""
    o = np.asarray(obs, np.float32)
    return mirror_frames(o[..., [2, 3, 0, 1], :])
