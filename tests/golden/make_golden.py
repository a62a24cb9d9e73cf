#!/usr/bin/env python
"""Generates tests/golden/step_v2.npz: 256 seeded env states of the four scenario kinds of tests/parity_util.py
(open field, wall / corner / goal-mouth huggers, scrums, ball crossing a goal line), two consecutive steps with
out-of-range actions, and everything the step produces (body state, bias velocities, counters, stacked observations,
rewards, done / goal flags, the arbiter cache with its accumulated impulses) plus the poses behind the two
history frames of every state (the simulator keeps its observation history as poses, include/msoc.h).

The vectors come from the CPU oracle (oracle/soccer_oracle.c), NOT from the reference itself: the reference is pure
Python over pymunk, which cannot be imported or installed in this environment (DESIGN.md section 2: parity
unpinned at the pymunk boundary).  They freeze the oracle's behaviour, so that a change to the oracle, to the host
build of the kernel arithmetic or to the kernels shows up against a fixed file.

    python tests/golden/make_golden.py        (from the repo root; rewrites the .npz)
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
import golden_util as G  # noqa: E402
import oracle_lib as O  # noqa: E402
import parity_util as P  # noqa: E402

N, SEED = 256, 20261018
rng = np.random.default_rng(SEED)
states0 = [P.random_state(rng, P.KINDS[i % 4]) for i in range(N)]
ora = O.OracleVec(N, P.CONFIG, seed=0)
ora.set_states(states0)
hist0 = [s["hist"] for s in states0]
states0 = ora.get_states()  # as the oracle holds them
for s, h in zip(states0, hist0):
    s["hist"] = h  # the poses behind the two frames of the injected history (the oracle itself keeps frames)
act1 = rng.uniform(-1.2, 1.2, (N, 4, 3)).astype(np.float32)
act2 = rng.uniform(-1.2, 1.2, (N, 4, 3)).astype(np.float32)
o1, r1, d1, g1 = ora.step(act1, auto_reset=False)
states1 = ora.get_states()
for s, s0 in zip(states1, states0):
    s["hist"] = [s0["hist"][1], P.pose_of(s)]  # after the step: the older injected pose and the state itself
o2, r2, d2, g2 = ora.step(act2, auto_reset=False)
states2 = ora.get_states()
for s, s1 in zip(states2, states1):
    s["hist"] = [s1["hist"][1], P.pose_of(s)]
out = {"act1": act1, "act2": act2, "rew1": r1, "rew2": r2, "done1": d1, "done2": d2, "goal1": g1, "goal2": g2}
for name, st in (("s0", states0), ("s1", states1), ("s2", states2)):
    out.update(G.pack(st, name))
# the observation a step returns is the one its state holds: stored once, as s1_obs / s2_obs
assert np.array_equal(o1, out["s1_obs"]) and np.array_equal(o2, out["s2_obs"])
path = os.path.join(HERE, "step_v2.npz")
G.save(path, out)
nc = sum(len(s["cache"]) for s in states1)
print(f"wrote {path}: {N} envs, {int(np.abs(g1).sum())}+{int(np.abs(g2).sum())} goals, {nc} cached arbiters after step 1, "
      f"{os.path.getsize(path) / 1e3:.0f} kB")
