"""One handle driven through every entry point in turn -- msoc_step, msoc_step_teams, MSOC_STEP_GENERAL_PATH, the replay
of a captured graph, the chunked host-buffer steps msoc_step_host / msoc_step_host_frames, a masked msoc_reset,
msoc_load_states and msoc_render -- against a twin handle that does every step as an eager msoc_step with the same
flags (bit for bit after every call), against the fp64 oracle on a sample of envs, and on the checked build.

The calls share the handle's control block: a whole step at step counter s takes its work-list counters from set s & 1
and relies on them being zero, and a host step of 131 072 envs or more runs in chunks with counters of their own.  The
sizes below are one chunk (the unchunked host path), three chunks with a ragged last one, and the eight-chunk cap."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import oracle_lib as O
import parity_util as P
from marl_soccer_b200 import _capi
from marl_soccer_b200.sim import BatchedSoccerSim

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEV = torch.device("cuda:0")
# short episodes: truncations and auto-resets fall inside the script
CFG = {**P.CONFIG, "simulation": {"max_steps": 9}}

# Every host step (msoc_step_host / _frames) follows a device-side step or replay, so each whole step after one starts on
# the list-counter set that the whole step before the host step used.  "capture" records three steps of the handle into
# a CUDA graph without running them (after the first load, which allocates the handle's injection array); "replay" runs
# them: three steps, an odd number, so the parity of the step counter changes across it.
SCRIPT = ("dev", "host", "dev", "host", "teams", "host", "general", "load", "host", "capture", "replay", "host",
          "reset", "host", "frames", "frames", "render", "dev", "host", "replay", "teams", "load", "host", "general",
          "host", "dev")
STEPS = {"dev": 1, "host": 1, "frames": 1, "teams": 1, "general": 1, "replay": 3}
GRAPH_STEPS = 3


def chunk_ranges(n):
    """The env ranges of the pipeline chunks of a host step of n envs (step_host_impl in msoc.cu)."""
    chunks = min(max(n // 65536, 1), 8)
    per = ((n + chunks - 1) // chunks + 127) & ~127
    return [(e0, min(e0 + per, n)) for e0 in range(0, n, per)]


def placements(rng, m):
    """(m, 5, 2) float32 body positions, no two bodies touching (agents are 30 x 30 boxes, the ball has radius 10), and
    (m, 2) ball velocities or NaN (keep the env's own).  Every fourth ball sits in a goal mouth and crosses the goal line
    in the next step (both goals alternately); the other bodies are well inside the field."""
    pos = np.zeros((m, 5, 2), np.float32)
    ball_vel = np.full((m, 2), np.nan, np.float32)
    for k in range(m):
        while True:
            p = np.stack([rng.uniform(45, 755, 5), rng.uniform(45, 555, 5)], axis=1)
            if k % 4 == 0:
                left = k % 8 == 0
                p[4] = (10.0 + rng.uniform(0.5, 2.5) if left else 790.0 - rng.uniform(0.5, 2.5), rng.uniform(250, 350))
                ball_vel[k] = ((-1.0 if left else 1.0) * rng.uniform(150, 200), rng.uniform(-20, 20))
            d = np.linalg.norm(p[:, None] - p[None], axis=-1) + np.eye(5) * 1e3
            if d.min() > 45.0:
                break
        pos[k] = p
    return pos, ball_vel


class Plan:
    """What the script touches at size n, drawn from a seed before it runs: the envs of the two loads (a few hundred each,
    among them the envs on both sides of every chunk boundary), their new body positions and the balls sent into a goal,
    the envs rendered and the reset mask."""

    def __init__(self, n, seed):
        rng = np.random.default_rng(seed)
        self.n = n
        self.chunks = chunk_ranges(n)
        edges = [e0 for e0, _ in self.chunks[1:]] + [0, n - 1, n]
        near = {e + d for e in edges for d in (-2, -1, 0, 1) if 0 <= e + d < n}
        self.loads = []
        for _ in range(2):
            idx = np.unique(np.concatenate([np.fromiter(near, np.int64), rng.choice(n, 240, replace=False)]))
            self.loads.append((idx, *placements(rng, idx.size)))
        self.render_idx = np.unique(np.concatenate([np.fromiter(near, np.int64), rng.choice(n, 16, replace=False)]))
        self.reset_mask = torch.from_numpy((np.arange(n) % 7 == 3).astype(np.uint8)).to(DEV)

    def oracle_sample(self, size, seed):
        """About `size` envs: the first and last 64 of every chunk, every env of the loads, the rest random."""
        rng = np.random.default_rng(seed)
        parts = [np.arange(e0, min(e0 + 64, e1)) for e0, e1 in self.chunks]
        parts += [np.arange(max(e1 - 64, e0), e1) for e0, e1 in self.chunks]
        parts += [idx for idx, _, _ in self.loads]
        base = np.unique(np.concatenate(parts))
        draw = rng.choice(self.n, size, replace=False)
        rest = draw[~np.isin(draw, base)][:max(size - base.size, 0)]
        return np.unique(np.concatenate([base, rest]))


class SampleOracle:
    """The fp64 oracle for a sorted list of env indices: one OracleVec per run of consecutive indices, created with the
    run's global offset, so that the spawn draws after a goal or a truncation (keyed by the global env index) are the
    device's."""

    def __init__(self, idx, config):
        cuts = np.flatnonzero(np.diff(idx) != 1) + 1
        self.runs = []
        for k0, k1 in zip(np.concatenate([[0], cuts]), np.concatenate([cuts, [idx.size]])):
            self.runs.append((int(k0), int(k1), O.OracleVec(int(k1 - k0), config, seed=0, global_offset=int(idx[k0]))))
        self._env = [(vec, k - k0) for k0, k1, vec in self.runs for k in range(k0, k1)]

    def env(self, i):
        vec, j = self._env[i]
        return vec.env(j)

    def set_states(self, states):
        for k0, k1, vec in self.runs:
            vec.set_states(states[k0:k1])

    def step(self, actions, auto_reset=True):
        outs = [vec.step(actions[k0:k1], auto_reset=auto_reset) for k0, k1, vec in self.runs]
        return tuple(np.concatenate(part) for part in zip(*outs))


class SampleRows:
    """get_states of a sample of a sim's envs under the sample's own numbering (what P.compare_all reads)."""

    def __init__(self, sim, idx):
        self.sim, self.idx = sim, idx

    def get_states(self, k):
        return self.sim.get_states(self.idx[np.asarray(k)])


class HostOut:
    """Host output buffers of msoc_step_host / msoc_step_host_frames, filled with values no step writes before every
    call, so that a range the copies miss shows."""

    def __init__(self, n):
        self.obs = np.empty((n, 4, 66), np.float32)
        self.frames = np.empty((n, 4, 22), np.float32)
        self.reward = np.empty((n, 2), np.float32)
        self.done = np.empty((n,), np.uint8)
        self.goal = np.empty((n,), np.int8)
        self.score = np.empty((n, 2), np.int32)

    def poison(self):
        for a, v in ((self.obs, np.nan), (self.frames, np.nan), (self.reward, np.nan), (self.done, 0xAB),
                     (self.goal, 0x55), (self.score, -7)):
            a.fill(v)


def _dev(x):
    return torch.from_numpy(x).to(DEV)


def _same_outputs(a, ref, what):
    for name in ("obs", "reward", "done", "goal", "score"):
        assert torch.equal(getattr(a, name), getattr(ref, name)), (what, name)
    if a.reward4 is not None and ref.reward4 is not None:
        assert torch.equal(a.reward4, ref.reward4), (what, "reward4")
    assert a.class_counts() == ref.class_counts(), (what, a.class_counts(), ref.class_counts())


def run_script(n, twin=True, oracle_size=0, seed=7):
    """Runs SCRIPT on handle A, and its steps as eager msoc_step / msoc_step_teams calls with the same flags on a twin
    handle B (twin=True): after every call, A's outputs (and the host buffers of a host step) must equal B's bit for
    bit; at the end their saved states and statistics.  oracle_size > 0: before every single step of A, the states of
    a sample of envs are read from A and stepped on the fp64 oracle with the same actions; A's results must agree
    within the oracle bands.  Returns a summary (coverage, statistics, oracle margins)."""
    L = _capi.lib()
    plan = Plan(n, seed)
    a = BatchedSoccerSim(n, config=CFG, device=DEV, seed=seed)
    b = BatchedSoccerSim(n, config=CFG, device=DEV, seed=seed) if twin else None
    sims = [s for s in (a, b) if s is not None]
    ref = b if twin else a  # what A is compared with, and where coverage is counted
    for s in sims:
        s.reset(_capi.MODE_FULL_RANDOM, seed=seed + 1)
    if twin:
        _same_outputs(a, b, "reset")
    gen = torch.Generator(device=DEV).manual_seed(seed)
    out = HostOut(n)
    graph, static = None, [torch.zeros((n, 4, 3), device=DEV) for _ in range(GRAPH_STEPS)]
    cov = {"goals_blue": 0, "goals_red": 0, "truncations": 0, "light": 0, "heavy": 0, "pair": 0, "multi": 0}
    sample = plan.oracle_sample(oracle_size, seed + 2) if oracle_size else None
    ora = SampleOracle(sample, CFG) if oracle_size else None
    st = torch.from_numpy(sample).to(DEV) if oracle_size else None
    orc = {"env_steps_compared": 0, "out_of_band": [], "worst": {}, "knife_edge_excluded": 0}
    loads = iter(plan.loads)
    steps = 0

    def count(sim):
        cov["goals_blue"] += int((sim.goal > 0).sum())
        cov["goals_red"] += int((sim.goal < 0).sum())
        cov["truncations"] += int(sim.done.sum())
        for k, v in sim.class_counts().items():
            cov[k] += v

    def host_step(act, frames):
        out.poison()
        fn = L.msoc_step_host_frames if frames else L.msoc_step_host
        _capi.check(fn(a._h, act.ctypes.data, (out.frames if frames else out.obs).ctypes.data, out.reward.ctypes.data,
                       out.done.ctypes.data, out.goal.ctypes.data, out.score.ctypes.data, _capi.STEP_AUTO_RESET,
                       a._stream()))

    for t, op in enumerate(SCRIPT):
        what = f"call {t} ({op}) at {n} envs"
        if op in ("dev", "host", "frames", "teams", "general"):
            act = torch.rand((n, 4, 3), generator=gen, device=DEV) * 2.4 - 1.2  # out-of-range actions are clipped
            if ora is not None:
                synced = [P.dev_to_oracle_state(s, o) for s, o in zip(a.get_states(sample), a.obs[st].cpu().numpy())]
                ora.set_states(synced)
                edge = P.goal_knife_edge(synced)
            stack = a.obs.cpu().numpy() if op == "frames" else None
            if op in ("host", "frames"):
                host_step(act.cpu().numpy(), op == "frames")
            else:
                a.step(act, team_rewards=op == "teams", general_path=op == "general")
            if twin:
                b.step(act, team_rewards=op == "teams", general_path=op == "general")
            steps += 1
            count(ref)
            if op == "host":
                assert torch.equal(_dev(out.obs), ref.obs), what
            if op == "frames":  # the caller's 3-frame stack, rebuilt from the newest frames (soccer_env.py:130-140, :92-96)
                s4 = stack.reshape(n, 4, 3, 22)
                s4[:, :, 0], s4[:, :, 1], s4[:, :, 2] = s4[:, :, 1].copy(), s4[:, :, 2].copy(), out.frames
                fresh = out.done.astype(bool)
                s4[fresh] = out.frames[fresh][:, :, None, :]
                assert torch.equal(_dev(stack), ref.obs), what
            if op in ("host", "frames"):
                for h, d in ((out.reward, ref.reward), (out.done, ref.done), (out.goal, ref.goal), (out.score, ref.score)):
                    assert torch.equal(_dev(h), d), what
            if ora is not None:
                o_o, r_o, d_o, g_o = ora.step(act[st].cpu().numpy(), auto_reset=True)
                o_d = out.obs[sample] if op == "host" else a.obs[st].cpu().numpy()
                r_d = (a.reward4[st, :2] if op == "teams" else a.reward[st]).cpu().numpy()
                assert np.array_equal(a.done[st].cpu().numpy(), d_o), what
                assert np.array_equal(a.goal[st].cpu().numpy()[~edge], g_o[~edge]), what
                worst, failing, cache_bad = P.compare_all(SampleRows(a, sample), ora, o_d, o_o, r_d, r_o, sample.size, skip=edge)
                assert not cache_bad, f"{what}: counters or arbiter cache differ from the oracle for envs {sample[cache_bad[:10]]}"
                orc["env_steps_compared"] += int((~edge).sum())
                orc["knife_edge_excluded"] += int(edge.sum())
                orc["out_of_band"] += [(t, int(sample[i]), d) for i, d in failing]
                for k, v in worst.items():
                    orc["worst"][k] = max(orc["worst"].get(k, 0.0), v)
        elif op == "load":  # moved bodies without history (hist_valid = 0): the next step starts from injected records
            idx, pos, ball_vel = next(loads)
            rec = a.save_states(idx).cpu().numpy().copy()
            arr = rec.view(_capi.ENV_STATE_DTYPE).reshape(-1)
            arr["pos"] = pos
            goal = ~np.isnan(ball_vel[:, 0])
            arr["vel"][goal, 4] = ball_vel[goal]
            arr["vbias"] = 0.0
            arr["wbias"] = 0.0
            arr["cache_count"] = 0
            arr["hist_valid"] = 0
            for s in sims:
                s.load_states(idx, torch.from_numpy(rec))
        elif op == "capture":
            torch.cuda.synchronize()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                for x in static:
                    a.step(x)
        elif op == "replay":
            for x in static:
                x.copy_(torch.rand((n, 4, 3), generator=gen, device=DEV) * 2.4 - 1.2)
            graph.replay()
            for x in static:
                if twin:
                    b.step(x)
                    count(b)
            if not twin:
                count(a)
            steps += GRAPH_STEPS
        elif op == "reset":
            for s in sims:
                s.reset(_capi.MODE_RANDOM, mask=plan.reset_mask)
        elif op == "render":  # draws, and changes nothing
            before, obs = a.save_states(), a.obs.clone()
            img = a.render(plan.render_idx, 36, 48)
            torch.cuda.synchronize()
            assert img.shape == (plan.render_idx.size, 36, 48, 3) and int(img.max()) > 0
            assert torch.equal(a.save_states(), before) and torch.equal(a.obs, obs), what
        if twin:
            _same_outputs(a, b, what)
    assert steps == sum(STEPS.get(op, 0) for op in SCRIPT)
    sa = a.stats()
    summary = {"envs": n, "chunks": len(plan.chunks), "steps": steps, "coverage": cov, "stats": sa}
    assert sa["env_steps"] == steps * n and sa["contact_overflow"] == 0 and sa["nonfinite_actions"] == 0, sa
    if twin:
        assert torch.equal(a.save_states(), b.save_states())
        sa, sb = dict(sa), b.stats()
        # the fp64 return sum is added with atomics in no fixed order (from fp32 warp sums of returns below ~10 here)
        assert sa.pop("episode_return_sum") == pytest.approx(sb.pop("episode_return_sum"), rel=1e-6, abs=1e-6 * sb["episodes"])
        assert sa == sb, (sa, sb)
    if ora is not None:
        summary["oracle"] = {"sample": int(sample.size), "env_steps_compared": orc["env_steps_compared"],
                             "knife_edge_goal_cases_excluded": orc["knife_edge_excluded"],
                             "out_of_band": len(orc["out_of_band"]), "out_of_band_examples": orc["out_of_band"][:5],
                             "worst_violation_ratio": {k: round(float(v), 3) for k, v in orc["worst"].items()}}
    for s in sims:
        s.close()
    return summary


@pytest.mark.parametrize("n", [131071, 200003, 589825])
def test_mixed_entry_points_equal_a_device_only_twin(n):
    """One chunk (the control: the host step is a whole step), three chunks (the last one ragged: 66 627 envs, not
    a multiple of 32) and the eight-chunk cap."""
    assert len(chunk_ranges(n)) == {131071: 1, 200003: 3, 589825: 8}[n]
    s = run_script(n)
    cov = s["coverage"]
    print(f"mixed sequence at {n} envs ({s['chunks']} chunks, {s['steps']} steps): coverage {cov}")
    P.record(f"sequences/mixed_vs_twin_{n}", {"chunks": s["chunks"], "steps": s["steps"], "coverage": cov})
    assert all(v > 0 for v in cov.values()), cov  # goals of both sides, truncations and every contact class


def test_mixed_entry_points_match_the_fp64_oracle():
    """The same calls on one handle, without a twin: ~1 500 envs (both ends of every chunk, the loaded envs, random
    ones) are stepped on the oracle from the device's states before each step, within the tracked-rollout slack."""
    n = 200003
    s = run_script(n, twin=False, oracle_size=1500)
    o = s["oracle"]
    worst = max(o["worst_violation_ratio"].values())
    print(f"mixed sequence vs the oracle at {n} envs: {o}, coverage {s['coverage']}, worst ratio {worst}")
    P.record("sequences/mixed_vs_oracle", {**o, "coverage": s["coverage"]})
    single = sum(op in STEPS and op != "replay" for op in SCRIPT)
    assert o["env_steps_compared"] + o["knife_edge_goal_cases_excluded"] == single * o["sample"] and o["sample"] >= 1400, o
    assert o["out_of_band"] <= o["env_steps_compared"] * P.MAX_TRACKED_FRACTION, o
    assert worst < P.MAX_RATIO, o


CHECKED = r"""
import sys
sys.path.insert(0, %(root)r); sys.path.insert(0, %(root)r + "/tests")
from marl_soccer_b200 import _capi
import test_gpu_sequences as S
L = _capi.lib()
assert L.msoc_debug_errors() == 0, "checks are compiled in and clean at start"
s = S.run_script(200003)
bits = L.msoc_debug_errors()
assert bits == 0, bin(bits)
assert s["stats"]["contact_overflow"] == 0, s
print("checked sequence clean", s["coverage"])
"""


def test_mixed_entry_points_on_the_checked_build():
    """The twin comparison at three chunks on libmsoc_checked.so: no list count or list entry outside the
    stepped range (CHK_LIST_COUNT, CHK_LIST_ENV), nor any other of the kernels' own checks."""
    from marl_soccer_b200 import build
    env = dict(os.environ, MSOC_LIB=build.build_checked())
    r = subprocess.run([sys.executable, "-c", CHECKED % {"root": ROOT}], env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "checked sequence clean" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]
    print(r.stdout.strip().splitlines()[-1])
