#!/usr/bin/env python
"""Cost of red's own reward (msoc_step_teams) and of the shared-policy self-play rollout on one GPU, with the card's
name, power limit and max SM clock read in the same run.

    python tools/team_bench.py [--out profiles/r06_teams.json]

(a) msoc_step against msoc_step_teams on two handles with the same seed and actions, at 65 536 and 1 Mi envs: CUDA
    events, windows of back-to-back auto-reset steps with fresh U(-1, 1) actions (a seeded pool of 16, cycled) after a
    200-step pre-roll, the two calls alternated window by window, best and mean.  The envs' records (1 741 B of
    traffic per env-step) are larger than L2 at 1 Mi envs, not at 65 536.
(b) BASELINE config 5: 262 144 envs x 128 steps, bf16 GraphedRollout, with blue learning alone against U(-1, 1), with a
    one-slot bf16 Opponent, and with self_play=True (one policy, both teams learn): ms per rollout step, env-steps/s and
    learning env-agent-steps/s (2 trained rows per env-step, 4 with self-play).  The three graphs are replayed
    alternately in one process."""
from __future__ import annotations

import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from marl_soccer_b200 import _capi  # noqa: E402
from marl_soccer_b200.rollout import Agent, GraphedRollout, RolloutBuffer, RunningMeanStd  # noqa: E402
from marl_soccer_b200.selfplay import Opponent  # noqa: E402
from marl_soccer_b200.sim import BatchedSoccerSim, load_default_config  # noqa: E402
from state_bench import gpu_info  # noqa: E402

ACTION_POOL = 16  # seeded action tensors cycled by the step timing
PREROLL = 200     # steps of each handle before the first timed window


def step_case(n: int, steps: int, windows: int) -> dict:
    dev = torch.device("cuda:0")
    sims = {k: BatchedSoccerSim(n, config=load_default_config(), device=dev, seed=0) for k in ("step", "step_teams")}
    for s in sims.values():
        s.reset(_capi.MODE_FULL_RANDOM, seed=0)
    # fresh U(-1, 1) actions every step, cycled from a seeded pool (one action held for every step piles the agents
    # into the walls and measures the contact kernel's worst case instead)
    g = torch.Generator(device=dev).manual_seed(0)
    pool = [torch.rand((n, 4, 3), generator=g, device=dev) * 2.0 - 1.0 for _ in range(ACTION_POOL)]
    calls = {"step": lambda a: sims["step"].step(a), "step_teams": lambda a: sims["step_teams"].step(a, team_rewards=True)}
    for fn in calls.values():  # warm-up (module load, the (N, 4) reward allocation) and a pre-roll into the step mix
        for t in range(PREROLL):
            fn(pool[t % ACTION_POOL])
    times = {k: [] for k in calls}
    t0 = PREROLL
    for _ in range(windows):  # both handles see the same actions in the same order: they hold the same states
        for k, fn in calls.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for t in range(t0, t0 + steps):
                fn(pool[t % ACTION_POOL])
            e1.record()
            torch.cuda.synchronize()
            times[k].append(e0.elapsed_time(e1) / steps)
        t0 += steps
    out = {"envs": n, "steps_per_window": steps, "windows": windows}
    for k, ts in times.items():
        out[k] = {"ms_best": round(min(ts), 4), "ms_mean": round(sum(ts) / len(ts), 4)}
    out["teams_over_step_best"] = round(min(times["step_teams"]) / min(times["step"]), 4)
    out["teams_over_step_mean"] = round(sum(times["step_teams"]) / sum(times["step"]), 4)
    return out


def rollout_case(n: int, T: int, windows: int) -> dict:
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    agent = Agent().to(dev)
    rms = RunningMeanStd((66,), dev)
    variants = {}
    for k in ("blue_only", "opponent_1_slot", "self_play"):
        sim = BatchedSoccerSim(n, config=load_default_config(), device=dev, seed=0)
        sim.reset(_capi.MODE_FULL_RANDOM, seed=0)
        buf = RolloutBuffer(T, n, dev, obs_dtype=torch.bfloat16, agents=4 if k == "self_play" else 2)
        opp = None
        if k == "opponent_1_slot":
            opp = Opponent(n, slots=1, device=dev, policy_dtype=torch.bfloat16)
            opp.set(0, agent, rms)
        variants[k] = GraphedRollout(sim, agent, rms, buf, policy_dtype=torch.bfloat16, opponent=opp,
                                     self_play=k == "self_play")
    for ro in variants.values():
        ro.run()  # eager warm-up + capture
        ro.run()  # one replay
    times = {k: [] for k in variants}
    for _ in range(windows):
        for k, ro in variants.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            ro.run()
            e1.record()
            torch.cuda.synchronize()
            times[k].append(e0.elapsed_time(e1))
    out = {"envs": n, "steps": T, "windows": windows}
    for k, ts in times.items():
        best, mean = min(ts) / T, sum(ts) / len(ts) / T
        rows = 4 if k == "self_play" else 2
        out[k] = {"ms_per_step_best": round(best, 4), "ms_per_step_mean": round(mean, 4),
                  "env_steps_per_s_best": round(n / best * 1e3),
                  "learning_env_agent_steps_per_s_best": round(rows * n / best * 1e3)}
    return out


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--windows", type=int, default=6)
    ap.add_argument("--envs", type=int, default=262144)
    ap.add_argument("--rollout-steps", type=int, default=128)
    ap.add_argument("--rollout-windows", type=int, default=4)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("team_bench.py needs a CUDA device")
    result = {**gpu_info(), "step": [step_case(n, args.steps, args.windows) for n in (65536, 1 << 20)]}
    print(json.dumps(result["step"]), flush=True)
    result["rollout"] = rollout_case(args.envs, args.rollout_steps, args.rollout_windows)
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
