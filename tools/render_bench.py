#!/usr/bin/env python
"""Device rendering throughput (msoc_render) on one GPU, with the two numbers it is judged against taken in the same
process: the write rate of a zero_() of a uint8 buffer of the same size (the ceiling of a write-only kernel), and the
step time at the same env count.  Every output is larger than the 126 MB L2, so the timed calls write to HBM.

    python tools/render_bench.py [--calls 50] [--out FILE]

States come from a staggered pre-roll with random actions (env i re-spawned at step i % 100), so the agents are
rotated, in contact and spread over the field as in training."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from marl_soccer_b200.sim import BatchedSoccerSim  # noqa: E402

WORKLOADS = [(65536, 84, 84), (65536, 96, 128), (262144, 64, 64), (4096, 600, 800)]


def timed(fn, calls: int, reps: int = 3) -> float:
    """Best of `reps` windows of `calls` back-to-back calls, ms per call (CUDA events)."""
    best = float("inf")
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(calls):
            fn()
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1) / calls)
    return best


def gpu_info() -> dict:
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in q.split(",")]
        info.update({"nvidia_smi_name": name, "power_limit": power, "max_sm_clock": clock})
    except Exception as e:  # the query is informative only
        info["nvidia_smi_error"] = str(e)
    return info


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--preroll", type=int, default=150)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("render_bench.py needs a CUDA device")
    result = {**gpu_info(), "calls": args.calls, "workloads": []}
    for n, H, W in WORKLOADS:
        sim = BatchedSoccerSim(n, seed=1)
        sim.reset(2, seed=2)
        g = torch.Generator(device="cuda").manual_seed(0)
        acts = torch.rand((8, n, 4, 3), generator=g, device="cuda") * 2 - 1
        ar = torch.arange(n, device="cuda")
        for t in range(args.preroll):
            sim.step(acts[t % 8])
            if t < 100:
                sim.reset(2, mask=(ar % 100 == t))
        out = torch.empty((n, H, W, 3), dtype=torch.uint8, device="cuda")
        fill = torch.empty_like(out)
        for _ in range(args.warmup):
            sim.render(None, H, W, out=out)
            fill.zero_()
        bytes_out = out.numel()
        ms_render = timed(lambda: sim.render(None, H, W, out=out), args.calls)
        ms_fill = timed(lambda: fill.zero_(), args.calls)
        k = [0]

        def step():
            sim.step(acts[k[0] % 8])
            k[0] += 1
        for _ in range(args.warmup):
            step()
        ms_step = timed(step, args.calls)
        row = {"envs": n, "height": H, "width": W, "bytes_per_call": bytes_out,
               "render_ms": round(ms_render, 4), "render_gbs": round(bytes_out / ms_render / 1e6, 1),
               "fill_ms": round(ms_fill, 4), "fill_gbs": round(bytes_out / ms_fill / 1e6, 1),
               "fraction_of_fill_rate": round(ms_fill / ms_render, 3), "step_ms": round(ms_step, 4)}
        print(json.dumps(row), flush=True)
        result["workloads"].append(row)
        del out, fill, acts
        sim.close()
        torch.cuda.empty_cache()
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
