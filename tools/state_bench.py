#!/usr/bin/env python
"""Throughput of msoc_save_states / msoc_load_states (BatchedSoccerSim.save_states, load_states, clone_envs) on one GPU,
with the two numbers they are judged against taken in the same process: a copy_ of a uint8 buffer of the snapshot's
size (read + write, the ceiling of a kernel that moves each byte once) and one step at the same env count.

    python tools/state_bench.py [--envs 1048576] [--calls 20] [--out FILE]

States come from a staggered pre-roll with random actions (env i re-spawned at step i % 100), so the agents are rotated,
in contact, and carry bias blocks and arbiter-cache entries as in training.  Algorithmic bytes per env: the 808-byte
record, plus its two state records (256 B), score, seed and spawn count (20 B), plus the 64-byte bias block and 12 bytes
per cache entry where the snapshot says they exist -- counted from the snapshot itself."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from marl_soccer_b200 import _capi  # noqa: E402
from marl_soccer_b200.sim import BatchedSoccerSim  # noqa: E402


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


def algorithmic_bytes(snap: torch.Tensor) -> int:
    """Bytes a save or a load of these records has to move (module docstring)."""
    f = _capi.state_fields(snap)
    n = snap.shape[0]
    has_bias = ((f["vbias"] != 0).flatten(1).any(dim=1) | (f["wbias"] != 0).any(dim=1)).sum().item()
    entries = f["cache_count"].view(torch.int32).clamp(max=_capi.MAX_CACHE).sum().item()
    return n * (_capi.ENV_STATE_BYTES + 2 * 128 + 20) + 64 * has_bias + 12 * entries


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=1 << 20)
    ap.add_argument("--subset", type=int, default=1 << 16)
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--preroll", type=int, default=150)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("state_bench.py needs a CUDA device")
    n, m = args.envs, args.subset
    sim = BatchedSoccerSim(n, seed=1)
    sim.reset(2, seed=2)
    g = torch.Generator(device="cuda").manual_seed(0)
    acts = torch.rand((8, n, 4, 3), generator=g, device="cuda") * 2 - 1
    ar = torch.arange(n, device="cuda")
    for t in range(args.preroll):
        sim.step(acts[t % 8])
        if t < 100:
            sim.reset(2, mask=(ar % 100 == t))
    snap = sim.save_states()
    alg_all = algorithmic_bytes(snap)
    perm = torch.randperm(n, generator=g, device="cuda")
    sub_idx, dst_idx = perm[:m].contiguous(), perm[m:2 * m].contiguous()
    alg_sub = algorithmic_bytes(snap[sub_idx])
    sub = torch.empty((m, _capi.ENV_STATE_BYTES), dtype=torch.uint8, device="cuda")
    copy_src, copy_dst = torch.empty_like(snap), torch.empty_like(snap)

    cases = {
        "save_all": (lambda: sim.save_states(out=snap), alg_all),
        "load_all": (lambda: sim.load_states(None, snap), alg_all),
        "save_subset": (lambda: sim.save_states(sub_idx, out=sub), alg_sub),
        "load_subset": (lambda: sim.load_states(sub_idx, sub), alg_sub),
        # a clone is a save and a load of the same records plus the (N,4,66) observation rows, read and written
        "clone_subset": (lambda: sim.clone_envs(sub_idx, dst_idx), 2 * alg_sub + 2 * m * 4 * 66 * 4),
    }
    for fn, _ in cases.values():
        for _ in range(args.warmup):
            fn()
    for _ in range(args.warmup):
        copy_dst.copy_(copy_src)
    ms_copy = timed(lambda: copy_dst.copy_(copy_src), args.calls)
    copy_gbs = 2 * snap.numel() / ms_copy / 1e6
    k = [0]

    def step():
        sim.step(acts[k[0] % 8])
        k[0] += 1
    for _ in range(args.warmup):
        step()
    ms_step = timed(step, args.calls)
    result = {**gpu_info(), "envs": n, "subset": m, "calls": args.calls, "snapshot_bytes": snap.numel(),
              "algorithmic_bytes_all": alg_all, "algorithmic_bytes_subset": alg_sub,
              "copy_ms": round(ms_copy, 4), "copy_gbs": round(copy_gbs, 1), "step_ms": round(ms_step, 4), "cases": {}}
    for name, (fn, nbytes) in cases.items():
        ms = timed(fn, args.calls)
        gbs = nbytes / ms / 1e6
        row = {"ms": round(ms, 4), "algorithmic_bytes": nbytes, "gbs": round(gbs, 1),
               "fraction_of_copy_bandwidth": round(gbs / copy_gbs, 3)}
        print(json.dumps({name: row}), flush=True)
        result["cases"][name] = row
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
