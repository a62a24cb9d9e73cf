#!/usr/bin/env python
"""Cost of self-play on one GPU (marl_soccer_b200/selfplay.py), with the card's name, power limit and max SM clock read
in the same run.

    python tools/selfplay_bench.py [--out profiles/r05_selfplay.json]

(a) msoc_team_inputs team 1 (mirrored red rows) against team 0 and against msoc_policy_inputs, at 262 144 and 1 Mi envs,
    as the opponent calls it (policy input only: no raw copy, no moments).  CUDA events, best of three windows; the
    observation buffer (1 056 B per env) is larger than L2 at both sizes.  Bytes per call: 528 read + 264 written per
    env (2 rows x 66 bf16).
(b) BASELINE config 5: 262 144 envs x 128 steps, bf16 GraphedRollout, with red playing U(-1, 1), one opponent slot and
    four slots (bf16 Opponent), the three graphs replayed alternately in one process on one sim: ms per rollout step and
    env-steps/s, best and mean of the windows."""
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
from state_bench import gpu_info, timed  # noqa: E402


def kernel_case(n: int, calls: int) -> dict:
    L = _capi.lib()
    dev = torch.device("cuda:0")
    st = torch.cuda.current_stream(dev).cuda_stream
    obs = torch.randn((n, 4, 66), device=dev)
    shift, inv_std = torch.randn(66, device=dev), torch.rand(66, device=dev) + 0.5
    x72 = torch.zeros((2 * n, 72), dtype=torch.bfloat16, device=dev)
    calls_by_name = {
        "policy_inputs": lambda: L.msoc_policy_inputs(obs.data_ptr(), n, shift.data_ptr(), inv_std.data_ptr(), x72.data_ptr(), None, None, st),
        "team0": lambda: L.msoc_team_inputs(obs.data_ptr(), n, 0, shift.data_ptr(), inv_std.data_ptr(), x72.data_ptr(), None, None, st),
        "team1": lambda: L.msoc_team_inputs(obs.data_ptr(), n, 1, shift.data_ptr(), inv_std.data_ptr(), x72.data_ptr(), None, None, st),
    }
    for fn in calls_by_name.values():
        for _ in range(3):
            _capi.check(fn())
    nbytes = n * (2 * 66 * 4 + 2 * 66 * 2)
    best = {k: float("inf") for k in calls_by_name}
    for _ in range(3):  # alternate the three calls, best window of each
        for k, fn in calls_by_name.items():
            best[k] = min(best[k], timed(fn, calls, reps=1))
    row = {"envs": n, "bytes_per_call": nbytes}
    for k, ms in best.items():
        row[k] = {"ms": round(ms, 4), "gbs": round(nbytes / ms / 1e6, 1)}
    row["team1_over_team0"] = round(best["team1"] / best["team0"], 3)
    row["team1_over_policy_inputs"] = round(best["team1"] / best["policy_inputs"], 3)
    return row


def rollout_case(n: int, T: int, windows: int) -> dict:
    dev = torch.device("cuda:0")
    sim = BatchedSoccerSim(n, config=load_default_config(), device=dev, seed=0)
    sim.reset(_capi.MODE_FULL_RANDOM, seed=0)
    torch.manual_seed(0)
    agent = Agent().to(dev)
    rms = RunningMeanStd((66,), dev)
    buf = RolloutBuffer(T, n, dev, obs_dtype=torch.bfloat16)
    variants = {"red_random": None}
    for K in (1, 4):
        opp = Opponent(n, slots=K, device=dev, policy_dtype=torch.bfloat16)
        for k in range(K):
            opp.set(k, agent, rms)
        variants[f"opponent_{K}_slot{'s' if K > 1 else ''}"] = opp
    ros = {k: GraphedRollout(sim, agent, rms, buf, policy_dtype=torch.bfloat16, opponent=o) for k, o in variants.items()}
    for ro in ros.values():
        ro.run()  # eager warm-up + capture
        ro.run()  # one replay
    times = {k: [] for k in ros}
    for _ in range(windows):
        for k, ro in ros.items():
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
        out[k] = {"ms_per_step_best": round(best, 4), "ms_per_step_mean": round(mean, 4),
                  "env_steps_per_s_best": round(n / best * 1e3)}
    base = out["red_random"]["ms_per_step_best"]
    for k in times:
        out[k]["over_red_random"] = round(out[k]["ms_per_step_best"] / base, 3)
    return out


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=50)
    ap.add_argument("--envs", type=int, default=262144)
    ap.add_argument("--steps", type=int, default=128)
    ap.add_argument("--windows", type=int, default=4)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("selfplay_bench.py needs a CUDA device")
    result = {**gpu_info(), "team_inputs": [kernel_case(n, args.calls) for n in (262144, 1 << 20)]}
    print(json.dumps(result["team_inputs"]), flush=True)
    result["rollout"] = rollout_case(args.envs, args.steps, args.windows)
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
