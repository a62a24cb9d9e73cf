#!/usr/bin/env python
"""bench.py -- env-steps/sec of the fused soccer step on N B200s (envs sharded by global env index, no per-step
collective), with the HBM roofline of the step, the end-to-end number through the host-buffer C-ABI calls, and the
CPU oracle timed on the host cores as the reported baseline.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--envs-per-gpu E | --global-envs G] [--impl reference]
                    [--dump-outputs DIR]

One "step" = one msoc_step call over this rank's shard = two kernel launches (the streaming contact-free kernel over
all envs, then one persistent contact kernel over the envs it declined, by work class).  Under torchrun (N > 1) every
rank owns a contiguous range of global env indices: E envs each by default (weak scaling, BASELINE config 4's total on
every GPU), or G / N with --global-envs G (strong scaling: BASELINE config 4 as written, 1 048 576 envs split over
2/4/8 GPUs).  At N = 1 the line also carries BASELINE config 3 (65 536 envs, eager and as a replayed CUDA graph) and
config 5 (PPO rollout with the MLP policy in the loop) as sub-records.

--dump-outputs DIR writes what the last timed step returned on rank 0 (see dump_outputs) as DIR/<name>.npy.  The
inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BYTES_PER_ENV_STEP = 2194  # SURVEY.md section 8(d): 940 B read + 1 254 B written, fp32, drop-in semantics
METRIC = "env_steps_per_sec"
UNIT = "env-steps/s"
DEFAULT_ENVS_PER_GPU = 1_048_576  # BASELINE config 4's total (1 Mi envs); working set >> 126 MB L2
DUMP_ENVS = 32768  # envs sampled for --dump-outputs: 1 088 B each over the six files, 36 MB in all
WORKLOAD = ("2v2 soccer, {n} envs per GPU ({g} in all), config.json defaults, i.i.d. random actions U(-1,1) (random "
            "windows of a pre-generated device buffer), auto-reset in full-random mode, shaped rewards, episodes "
            "staggered over all phases")


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def recorded_traffic():
    """dram bytes per step (sum over the step kernels) from the committed ncu capture, or None."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            return json.load(f)
    except Exception:
        return None


class ClockSampler(threading.Thread):
    """Samples nvidia-smi clocks / throttle reasons while the timed region runs."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.samples, self._halt = index, [], threading.Event()

    def run(self):
        while not self._halt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                      "-i", str(self.index)], capture_output=True, text=True, timeout=5).stdout
                parts = [x.strip() for x in out.strip().split(",")]
                if len(parts) >= 7:
                    self.samples.append(parts)
            except Exception:
                pass
            self._halt.wait(0.05)

    def stop(self):
        self._halt.set()
        self.join(timeout=6)
        sm = sorted(float(s[0]) for s in self.samples if s[0].replace(".", "").isdigit())
        mx = [float(s[1]) for s in self.samples if s[1].replace(".", "").isdigit()]
        reasons = set()
        for s in self.samples:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), s[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------ CPU arm
def cpu_oracle_run(n_envs: int, steps: int, threads: int, seed: int = 0):
    """Times the CPU oracle (oracle/liboracle.so, the restated reference path) on the host cores."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import numpy as np
    import oracle_lib as O
    vec = O.OracleVec(n_envs, O.DEFAULT_CONFIG, seed=seed)
    vec.reset(O.MODE_FULL_RANDOM, seed=seed)
    rng = np.random.default_rng(seed)
    flat = rng.uniform(-1, 1, 16 * n_envs * 12).astype(np.float32)  # i.i.d. windows, as on the GPU arm
    offs = rng.integers(0, 15 * n_envs, size=steps + 1) * 12
    vec.step(flat[offs[steps]:offs[steps] + n_envs * 12], auto_reset=True, nthreads=threads)
    t0 = time.perf_counter()
    for k in range(steps):
        vec.step(flat[offs[k]:offs[k] + n_envs * 12], auto_reset=True, nthreads=threads)
    dt = time.perf_counter() - t0
    return n_envs * steps / dt, dt


def cpu_dict_api_run(steps: int = 400):
    """BASELINE.md section 3.2 row (c): one env behind the reference's dict API (SoccerEnv.step with per-agent dicts,
    soccer_env.py:100-154) -- the Python overhead the reference pays on top of its physics, with the oracle as the
    physics."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import numpy as np
    import backends as B
    from marl_soccer_b200 import soccer_env
    env = soccer_env.soccerenv(_sim_factory=B.OracleBackedSim, _seed=1)
    env.reset(seed=0, options={"use_full_random_positions": True})
    rng = np.random.default_rng(0)
    acts = rng.uniform(-1, 1, (steps, 4, 3)).astype(np.float32)
    t0 = time.perf_counter()
    for k in range(steps):
        _, _, _, trunc, _ = env.step({f"agent_{i}": acts[k, i] for i in range(4)})
        if trunc["agent_0"]:
            env.reset()
    return steps / (time.perf_counter() - t0)


def reference_probe():
    """BASELINE.md section 3.1: the real reference is pure Python over pymunk / pygame / gymnasium / pettingzoo; when
    those import AND an unmodified copy of the reference is installed under baseline/_ref, its own soccerenv() is
    timed; otherwise (this image: none of the four is installable, no network) the oracle port stands in."""
    missing = []
    for m in ("pymunk", "pygame", "gymnasium", "pettingzoo"):
        try:
            __import__(m)
        except Exception:
            missing.append(m)
    ref_dir = os.path.join(ROOT, "baseline", "_ref", "soccer_simulation")
    if missing:
        return None, "not importable: " + ", ".join(missing)
    if not os.path.isdir(ref_dir):
        return None, "baseline/_ref/soccer_simulation is absent (the reference has no setup.py / pyproject.toml to install)"
    return ref_dir, "ok"


def real_reference_run(ref_dir: str, episodes: int = 3):
    """Times the unmodified reference: one SoccerEnv, full episodes of random actions, single process
    (the reference's vec env is a sequential loop over such envs, marl_vecenv.py:39)."""
    sys.path.insert(0, ref_dir)
    import numpy as np
    import soccer_env as ref_env  # the reference's own module
    env = ref_env.soccerenv()
    rng = np.random.default_rng(0)
    n = 0
    t0 = time.perf_counter()
    for ep in range(episodes):
        env.reset(seed=ep)
        done = False
        while not done:
            _, _, _, trunc, _ = env.step({a: rng.uniform(-1, 1, 3).astype(np.float32) for a in env.possible_agents})
            done = any(trunc.values())
            n += 1
    return n / (time.perf_counter() - t0)


def cpu_rows(cores: int):
    """BASELINE.md section 3.2: (a) 1 core, (b) all cores -- reported by the caller --, (c) behind the dict API."""
    rows = {}
    v, dt = cpu_oracle_run(256, 250, 1)
    rows["oracle_1_core"] = {"value": v, "unit": UNIT, "cores": 1, "sample": f"256 envs x 250 steps, {dt:.1f} s"}
    rows["oracle_dict_api_1_env"] = {"value": cpu_dict_api_run(400), "unit": UNIT, "cores": 1,
                                     "sample": "one env behind SoccerEnv's dict API (Python packaging per step), 400 steps"}
    return rows


def config_dict(n: int, world: int, preroll: int, scaling: str) -> dict:
    return {"workload": WORKLOAD.format(n=n, g=world * n), "envs_per_gpu": n, "global_envs": world * n, "scaling": scaling,
            "l2": "working set per GPU (three state buffers + obs + actions, ~1.7 KB/env) >> 126 MB L2; no flush needed",
            "preroll_steps": preroll}


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path on the host cores.  The real reference
    when it can run (reference_probe), else the oracle port (oracle/, the CPU restatement) on all host threads."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    n_gpu = args.global_envs // world if args.global_envs else args.envs_per_gpu
    scaling = "strong" if args.global_envs else "weak"
    ref_dir, why = reference_probe()
    if ref_dir is not None:
        value = real_reference_run(ref_dir)
        kind, used, sample = "reference", 1, "unmodified reference soccerenv(), 3 full episodes of random actions, single process"
        ms = 1e3 / value
    else:
        n_envs, per_step = 1024, 1000  # one bench "step" = one full 1000-step episode of 1024 envs (all phases)
        for _ in range(args.warmup):
            cpu_oracle_run(n_envs, 50, cores)
        t_total, k = 0.0, 0
        for _ in range(args.steps):
            _, dt = cpu_oracle_run(n_envs, per_step, cores)
            t_total += dt
            k += 1
        value = n_envs * per_step * k / t_total
        ms = 1e3 * t_total / max(1, k)
        kind, used = "port", cores
        sample = (f"oracle/liboracle.so (restated reference; the real one: {why}): {n_envs} envs x {per_step} steps per "
                  f"bench step, {k} bench steps, OpenMP over {cores} threads")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
        "higher_is_better": True, "scaling": scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": config_dict(n_gpu, world, args.preroll, scaling),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": used, "kind": kind, "sample": sample, "rows": cpu_rows(cores)},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------ GPU arm
def bind_near_gpu(torch, dev):
    """Pins this process to the CPUs NVML reports as local to the GPU (its NUMA node), so that the pinned host buffers
    of the end-to-end path are allocated next to the GPU's PCIe root.  Returns (previous affinity, CPUs bound) or
    (None, None) when NVML or the affinity call is unavailable."""
    try:
        import pynvml
        pynvml.nvmlInit()
        pr = torch.cuda.get_device_properties(dev)
        bus = "%08x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        h = pynvml.nvmlDeviceGetHandleByPciBusId(bus.encode())
        words = pynvml.nvmlDeviceGetCpuAffinity(h, ((os.cpu_count() or 64) + 63) // 64)
        cpus = [64 * i + b for i, w in enumerate(words) for b in range(64) if (int(w) >> b) & 1]
        old = os.sched_getaffinity(0)
        cpus = sorted(set(cpus) & set(old))
        if not cpus:
            return None, None
        os.sched_setaffinity(0, cpus)
        return old, len(cpus)
    except Exception:
        return None, None



def make_pool(torch, np, n, dev, seed, POOL=16):
    """Actions: one flat device buffer of 16*N*12 uniform(-1,1) floats generated before the timed region; step k reads
    the window starting at a pseudo-random env offset r_k, so every env sees an effectively i.i.d. action stream (a
    plain cycle over 16 tensors would give each env a periodic sequence with a constant net drift, pinning the agents
    against the walls)."""
    gen = torch.Generator(device=dev).manual_seed(1234 + seed)
    flat = torch.rand((POOL * n * 12,), generator=gen, device=dev) * 2 - 1
    offs = np.random.default_rng(99 + seed).integers(0, (POOL - 1) * n, size=1 << 16)

    class _Pool:
        def __getitem__(self, k):
            o = int(offs[k % len(offs)]) * 12
            return flat[o:o + n * 12].view(n, 4, 3)

        def window(self, k, g):
            """g consecutive action sets starting at a pseudo-random env offset (g <= POOL // 2)"""
            o = (int(offs[k % len(offs)]) % ((POOL - g) * n)) * 12
            return flat[o:o + g * n * 12].view(g, n, 4, 3)
    return _Pool()


def preroll(torch, sim, pool, cfg, steps, _capi):
    """Untimed: env i is re-spawned at pre-roll step hash(i) % max_steps, so after one episode length the episode
    phases are uniformly staggered and any timed window sees the time-average mix of spawn overlap, resting contacts,
    goals and auto-resets, whatever --steps is."""
    max_steps = int(cfg["simulation"]["max_steps"])
    phase = (torch.arange(sim.num_envs, device=sim.device, dtype=torch.int64) * 2654435761) % max_steps
    for k in range(steps):
        sim.reset(_capi.MODE_FULL_RANDOM, mask=(phase == (k % max_steps)))
        sim.step(pool[k])


def config3_record(torch, np, _capi, cfg, dev, peak):
    """BASELINE config 3: 65 536 envs on one GPU, auto-reset, shaped rewards.  The working set (~110 MB) sits in the
    126 MB L2, and the step is two short launches: eager launches expose the launch latency, a replayed CUDA graph
    of 20 steps (the device-side step counter makes any capture length replayable) shows the kernels themselves.
    The graph's steps read their actions from a static (20, N, 4, 3) buffer that is refilled with a fresh random window
    before every replay, inside the timed region: replaying the SAME action sets would give every env a periodic action
    sequence with a net drift, which pins the agents against the walls and multiplies the contact work (measured: a
    one-step graph replayed with constant actions takes 0.42 ms per step)."""
    from marl_soccer_b200.sim import BatchedSoccerSim
    n = 65536
    sim = BatchedSoccerSim(n, config=cfg, device=dev, seed=1)
    sim.reset(_capi.MODE_FULL_RANDOM, seed=1)
    pool = make_pool(torch, np, n, dev, 7, POOL=64)
    preroll(torch, sim, pool, cfg, 1000, _capi)
    K = 200
    for k in range(20):
        sim.step(pool[1000 + k])
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(K):
        sim.step(pool[1020 + k])
    e1.record()
    torch.cuda.synchronize(dev)
    eager_ms = e0.elapsed_time(e1) / K
    G = 20
    side = torch.cuda.Stream(device=dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side):
        for k in range(3):
            sim.step(pool[2000 + k])
    torch.cuda.current_stream(dev).wait_stream(side)
    acts = torch.empty((G, n, 4, 3), dtype=torch.float32, device=dev)
    acts.copy_(pool.window(2999, G))
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=side):
        for k in range(G):
            sim.step(acts[k])
    for r in range(3):
        acts.copy_(pool.window(3000 + r, G))
        graph.replay()
    torch.cuda.synchronize(dev)
    R = 20
    e0.record()
    for r in range(R):
        acts.copy_(pool.window(3100 + r, G))
        graph.replay()
    e1.record()
    torch.cuda.synchronize(dev)
    graph_ms = e0.elapsed_time(e1) / (R * G)
    st = sim.stats()
    del graph
    sim.close()
    return {"workload": "BASELINE config 3: 65 536 envs on one GPU, same action / episode-phase mix as the main line",
            "envs": n, "ms_per_step_eager": eager_ms, "ms_per_step_cuda_graph": graph_ms,
            "env_steps_per_s_eager": n / (eager_ms * 1e-3), "env_steps_per_s_cuda_graph": n / (graph_ms * 1e-3),
            "roofline_frac_cuda_graph": n * BYTES_PER_ENV_STEP / (graph_ms * 1e-3) / 1e9 / peak,
            "note": "working set fits the 126 MB L2: the HBM fraction is a comparison figure, not a bound",
            "contact_overflow": st["contact_overflow"]}


def config5_record(torch, _capi, cfg, dev, world_note="per GPU"):
    """BASELINE config 5: PPO self-play rollout loop, 262 144 envs x 128 steps with the reference's MLP policy in the
    loop (marl_soccer_b200/rollout.py), one GPU's shard."""
    from marl_soccer_b200.rollout import Agent, GraphedRollout, RolloutBuffer, RunningMeanStd
    from marl_soccer_b200.sim import BatchedSoccerSim
    n, T = 262144, 128
    sim = BatchedSoccerSim(n, config=cfg, device=dev, seed=2)
    torch.manual_seed(0)
    agent = Agent().to(dev)
    rms = RunningMeanStd((66,), dev)
    buf = RolloutBuffer(T, n, dev, obs_dtype=torch.bfloat16)
    sim.reset(_capi.MODE_FULL_RANDOM, seed=2)
    ro = GraphedRollout(sim, agent, rms, buf, policy_dtype=torch.bfloat16)
    ro.run()  # warm-up (captures the graph)
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    R = 2
    for _ in range(R):
        ro.run()
    e1.record()
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1)
    st = sim.stats()
    sim.close()
    return {"workload": f"BASELINE config 5: PPO rollout, {n} envs x {T} steps {world_note}, MLP policy (bf16, both nets packed into batched "
                        "GEMMs), normaliser (one fused pass per step) in the loop, one CUDA graph per rollout",
            "env_steps_per_s": n * T * R / (ms * 1e-3), "ms_per_rollout_step": ms / (T * R), "episodes": st["episodes"]}


def dump_outputs(torch, np, sim, offset: int, out_dir: str) -> None:
    """What the last step returned (obs, reward, done, goal, and the step's score) for a fixed, seeded sample of
    DUMP_ENVS envs, in env order, as float32 (the integer flags and counts are exact there), plus the global index of
    every sampled env (float64)."""
    n = sim.num_envs
    idx = np.sort(np.random.default_rng(0).choice(n, size=min(n, DUMP_ENVS), replace=False))
    sel = torch.from_numpy(idx).to(sim.device)
    os.makedirs(out_dir, exist_ok=True)
    for name in ("obs", "reward", "done", "goal", "score"):
        out = getattr(sim, name).index_select(0, sel).to(torch.float32).cpu().numpy()
        np.save(os.path.join(out_dir, f"{name}.npy"), out)
    np.save(os.path.join(out_dir, "env_index.npy"), (idx + offset).astype(np.float64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default 1000; --impl reference: 5)")
    ap.add_argument("--warmup", type=int, default=None, help="warm-up steps (default 100; --impl reference: 1)")
    ap.add_argument("--envs-per-gpu", type=int, default=DEFAULT_ENVS_PER_GPU)
    ap.add_argument("--global-envs", type=int, default=0, help="strong scaling: this many envs split over the GPUs")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--preroll", type=int, default=1000, help="untimed steps that decorrelate the episode phases")
    ap.add_argument("--e2e-steps", type=int, default=10)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the config-3 / config-5 sub-records")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned as DIR/<name>.npy")
    args = ap.parse_args()
    ref = args.impl == "reference"
    if args.steps is None:
        args.steps = 5 if ref else 1000  # a reference bench step is a whole 1000-step episode of 1024 envs on the CPU
    if args.warmup is None:
        args.warmup = 1 if ref else 100
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if ref:
        if args.dump_outputs:
            ap.error("--dump-outputs applies to the GPU path (--impl ours)")
        run_reference(args)
        return

    import numpy as np
    import torch
    from marl_soccer_b200 import _capi
    from marl_soccer_b200.sim import BatchedSoccerSim, load_default_config

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs CUDA devices (no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local_rank)
    dev = torch.device(f"cuda:{local_rank}")
    dist = None
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"  # keep stdout to the one JSON line (NCCL prints its version banner there)
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    scaling = "strong" if args.global_envs else "weak"
    if args.global_envs:
        from marl_soccer_b200.distributed import shard_range
        lo, hi = shard_range(args.global_envs, rank, world)
        n, offset = hi - lo, lo
    else:
        n, offset = args.envs_per_gpu, rank * args.envs_per_gpu
    cfg = load_default_config()
    L = _capi.lib()
    sim = BatchedSoccerSim(n, config=cfg, device=dev, seed=0, global_env_offset=offset)
    sim.reset(_capi.MODE_FULL_RANDOM, seed=0)
    pool = make_pool(torch, np, n, dev, rank)
    preroll(torch, sim, pool, cfg, args.preroll, _capi)
    W = max(3, args.warmup)
    for k in range(W):
        sim.step(pool[args.preroll + k])
    sim.stats(reset=True)
    torch.cuda.synchronize(dev)

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize(dev)
    launches0 = L.msoc_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    base_k = args.preroll + W
    for k in range(args.steps):
        sim.step(pool[base_k + k])
    stats_t = sim.stats_tensor(reset=False)
    if dist is not None:
        dist.all_reduce(stats_t)  # the only collective: one 64-byte sum per rollout
    e1.record()
    torch.cuda.synchronize(dev)
    if args.dump_outputs and rank == 0:
        dump_outputs(torch, np, sim, offset, args.dump_outputs)
    classes = sim.class_counts()  # work classes of the last timed step on this rank (instrumentation)
    if dist is not None:
        dist.barrier()
    elapsed_ms = e0.elapsed_time(e1)
    launches = L.msoc_launch_count() - launches0
    t = torch.tensor([elapsed_ms], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    elapsed_ms = float(t.item())
    # keep the GPU under the same load a little longer so that the clock sampler sees the timed workload
    if rank == 0:
        t_end = time.perf_counter() + 0.4
        k = 0
        while time.perf_counter() < t_end:
            sim.step(pool[base_k + args.steps + k]); k += 1
            if k % 50 == 0:
                torch.cuda.synchronize(dev)
        torch.cuda.synchronize(dev)
    clocks = sampler.stop() if rank == 0 else None
    stats = dict(zip([k for k, _ in _capi.MsocStats._fields_], stats_t.cpu().tolist()))
    total_envs = int(sum_over_ranks(torch, dist, dev, n))

    # device time of one step on this rank (two launches; events bracket K back-to-back steps)
    kernel_ms = e0.elapsed_time(e1) / args.steps
    value = total_envs * args.steps / (elapsed_ms * 1e-3)

    # end to end through the host-buffer C-ABI calls: pinned host actions in, pinned host results out, copies inside the
    # timed region.  Primary: msoc_step_host_frames (the newest frame per agent comes back, 352 B/env; the caller owns
    # the 3-frame stack as soccer_env.py:130-140 does).  Also: msoc_step_host (the full stacked observation).
    old_affinity, near_cpus = bind_near_gpu(torch, dev)
    h_acts = [torch.empty((n, 4, 3), dtype=torch.float32).pin_memory().copy_(pool[7 + j].cpu()) for j in range(4)]
    h_obs = torch.empty((n, 4, 66), dtype=torch.float32).pin_memory()
    h_frames = torch.empty((n, 4, 22), dtype=torch.float32).pin_memory()
    h_rew = torch.empty((n, 2), dtype=torch.float32).pin_memory()
    h_done = torch.empty((n,), dtype=torch.uint8).pin_memory()
    h_goal = torch.empty((n,), dtype=torch.int8).pin_memory()
    h_score = torch.empty((n, 2), dtype=torch.int32).pin_memory()
    stream = torch.cuda.current_stream(dev).cuda_stream

    def host_step_frames(j=0):
        _capi.check(L.msoc_step_host_frames(sim._h, h_acts[j % 4].data_ptr(), h_frames.data_ptr(), h_rew.data_ptr(),
                                            h_done.data_ptr(), h_goal.data_ptr(), h_score.data_ptr(), _capi.STEP_AUTO_RESET, stream))

    def host_step_full(j=0):
        _capi.check(L.msoc_step_host(sim._h, h_acts[j % 4].data_ptr(), h_obs.data_ptr(), h_rew.data_ptr(), h_done.data_ptr(),
                                     h_goal.data_ptr(), h_score.data_ptr(), _capi.STEP_AUTO_RESET, stream))

    def time_host(fn):
        for _ in range(3):
            fn()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        for j in range(args.e2e_steps):
            fn(j)
        torch.cuda.synchronize(dev)
        tt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if dist is not None:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return total_envs * args.e2e_steps / float(tt.item())
    e2e_frames = time_host(host_step_frames)
    e2e_full = time_host(host_step_full)
    if old_affinity is not None:
        os.sched_setaffinity(0, old_affinity)  # the CPU baseline below uses every core again
    h2d = n * 12 * 4
    small = n * (2 * 4 + 1 + 1 + 2 * 4)
    d2h_frames, d2h_full = n * 4 * 22 * 4 + small, n * 4 * 66 * 4 + small
    sim.close()

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    peak, peak_src = measured_peak()
    achieved = n * BYTES_PER_ENV_STEP / (kernel_ms * 1e-3) / 1e9
    traffic = recorded_traffic()
    extras = {}
    if world == 1 and not args.no_extras:
        try:
            extras["config3"] = config3_record(torch, np, _capi, cfg, dev, peak)
        except Exception as ex:  # a sub-record must never take the main line down
            extras["config3"] = {"error": repr(ex)}
        try:
            extras["config5_rollout"] = config5_record(torch, _capi, cfg, dev)
        except Exception as ex:
            extras["config5_rollout"] = {"error": repr(ex)}
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        steps_cpu = 1000  # one full episode: spawn overlap, contacts, truncation + auto-reset
        v, dt = cpu_oracle_run(4096, steps_cpu, cores)
        _, why = reference_probe()
        cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": f"oracle/liboracle.so (restated reference; the real one: {why}): 4096 envs x {steps_cpu} steps, "
                         f"OpenMP over {cores} threads, {dt:.1f} s",
               "rows": cpu_rows(cores)}
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": W,
        "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True, "scaling": scaling, "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": config_dict(n, world, args.preroll, scaling),
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": (traffic or {}).get("dram_bytes_per_launch_at_bench_size"),
                     "traffic_note": "DRAM bytes of one 1 Mi-env step from the committed ncu capture (profiles/traffic.json); below the "
                                     "algorithmic bytes because the observation history is rebuilt from 128-byte state records instead of read back",
                     "peak_source": peak_src, "algorithmic_bytes_per_env_step": BYTES_PER_ENV_STEP,
                     "kernel": "msoc_step = msoc_step_fast_kernel + msoc_step_contact_kernel "
                               "(whole step: algorithmic bytes of all envs / device time of the two launches)",
                     "kernel_ms": kernel_ms},
        "cpu_baseline": cpu,
        "e2e": {"value": e2e_frames, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h_frames,
                "steps": args.e2e_steps, "host_cpus_near_gpu": near_cpus, "api": "msoc_step_host_frames (pinned host buffers; newest frame per agent, the caller owns the stack)",
                "full_observation": {"value": e2e_full, "d2h_bytes_per_step": d2h_full, "api": "msoc_step_host ((N,4,66) stacked observation)"}},
        "gpu_launches": int(launches),
        "class_mix_last_step": {**{k: v / n for k, v in classes.items()}, "contact_free": 1.0 - sum(classes.values()) / n},
        "clocks": clocks,
        "stats": stats,
    }
    line.update(extras)
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


def sum_over_ranks(torch, dist, dev, n):
    t = torch.tensor([float(n)], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(t)
    return t.item()


if __name__ == "__main__":
    main()
