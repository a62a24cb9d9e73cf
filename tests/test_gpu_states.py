"""msoc_save_states / msoc_load_states on the device and the layers above them: the record format against get_states,
exact resume from a state_dict at every step-counter phase, resharding a checkpoint over handles, clone_envs, no side
effects, index handling, graph capture of a rewind loop, the NumPy path, and the checked build."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import parity_util as P
from marl_soccer_b200 import _capi
from marl_soccer_b200.host_api import HostBufferSim
from marl_soccer_b200.marl_vecenv import TorchSoccerVecEnv
from marl_soccer_b200.sim import BatchedSoccerSim

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CFG = {**P.CONFIG, "simulation": {"max_steps": 60}}
B = _capi.ENV_STATE_BYTES


def staggered_sim(n, seed=0, steps=90, offset=0):
    """n envs after a pre-roll with random actions and auto-reset; env i is re-spawned at step i % 60, so the episode
    phases are spread over the whole episode."""
    sim = BatchedSoccerSim(n, config=CFG, seed=seed, global_env_offset=offset)
    sim.reset(2, seed=seed + 1)
    g = torch.Generator(device="cuda").manual_seed(seed)
    ar = torch.arange(n, device="cuda")
    for t in range(steps):
        sim.step(torch.rand((n, 4, 3), generator=g, device="cuda") * 2 - 1)
        if t < 60:
            sim.reset(2, mask=(ar % 60 == t))
    return sim


def host_bytes(states):
    return np.frombuffer(b"".join(bytes(S) for S in states), np.uint8).reshape(len(states), B)


def outputs(sim):
    return [x.clone() for x in (sim.obs, sim.reward, sim.done, sim.goal, sim.score)]


def inject_some(sim, idx, shift=25.0):
    """set_states with hist_valid = 0 and moved bodies: the envs get a pending injected record (FLAG_INJECT)"""
    st = sim.get_states(idx)
    for k, S in enumerate(st):
        S.hist_valid = 0
        S.pos[k % 5][0] += shift
        S.ang[k % 4] = 0.3 * k
    sim.set_states(idx, st)


def test_format_matches_get_states_at_every_phase():
    n = 4096
    sim = staggered_sim(n, seed=3)
    inject_some(sim, [5, 77, 4095])
    g = torch.Generator(device="cuda").manual_seed(9)
    seen_bias = seen_cache = 0
    for phase in range(6):
        snap = sim.save_states()
        assert snap.shape == (n, B) and snap.dtype == torch.uint8 and snap.is_cuda
        want = host_bytes(sim.get_states(np.arange(n)))
        assert np.array_equal(snap.cpu().numpy(), want), phase
        f = _capi.state_fields(snap)
        assert bool((f["hist_valid"] == 1).all())
        seen_bias += int((f["vbias"] != 0).any(dim=2).any(dim=1).sum())
        seen_cache += int(f["cache_count"].view(torch.int32).sum())
        # save -> load -> save is a bitwise fixed point
        sim.load_states(None, snap)
        assert torch.equal(sim.save_states(), snap), phase
        # a subset, with repeats
        idx = [4095, 0, 5, 5, 1000]
        assert torch.equal(sim.save_states(idx), snap[idx])
        sim.step(torch.rand((n, 4, 3), generator=g, device="cuda") * 2 - 1)
    assert seen_bias > 0 and seen_cache > 0
    # fields against sources that do not go through the state kernels: the score and step counters (msoc_read_counters)
    # and the per-env seeds of the staggered reset (seed + 1 + global index; none of the envs was re-seeded since)
    f = _capi.state_fields(sim.save_states())
    score, steps = sim.counters()
    injected = [5, 77, 4095]
    mask = np.ones(n, bool); mask[injected] = False  # a pending injection's steps are in the injected record
    assert np.array_equal(f["score"].cpu().numpy(), score)
    assert np.array_equal(f["steps"].cpu().numpy()[mask], steps[mask])
    assert np.array_equal(f["seed"].cpu().numpy(), 4 + np.arange(n, dtype=np.uint64))
    # state_fields values are the ctypes fields
    snap = sim.save_states()
    f = {k: v.cpu().numpy() for k, v in _capi.state_fields(snap).items()}
    for i, S in zip([0, 5, 77, 4095], sim.get_states([0, 5, 77, 4095])):
        assert np.array_equal(f["pos"][i], np.array([[S.pos[b][0], S.pos[b][1]] for b in range(5)], np.float32))
        assert f["seed"][i] == S.seed and f["spawn_count"][i] == S.spawn_count and f["steps"][i] == S.steps
        assert f["cache_count"][i] == S.cache_count and list(f["cache_info"][i][:S.cache_count]) == list(S.cache_info)[:S.cache_count]
        assert np.array_equal(f["hist_ang"][i], np.array([list(S.hist_ang[0]), list(S.hist_ang[1])], np.float32))
    sim.close()


@pytest.fixture(scope="module")
def run_a():
    """Sim A (4 096 envs, max_steps 60, staggered): its state_dict, then 150 recorded steps."""
    n = 4096
    a = staggered_sim(n, seed=11)
    d = a.state_dict()
    stats0 = a.stats()
    g = torch.Generator(device="cuda").manual_seed(21)
    acts, outs, classes = [], [], []
    for _ in range(150):
        act = torch.rand((n, 4, 3), generator=g, device="cuda") * 2.2 - 1.1
        a.step(act)
        acts.append(act)
        outs.append(outputs(a))
        classes.append(a.class_counts())
    final = a.save_states()
    stats = a.stats()
    a.close()
    return {"n": n, "d": d, "stats0": stats0, "acts": acts, "outs": outs, "classes": classes, "final": final, "stats": stats}


def test_run_a_window_covers_resets_goals_and_contacts(run_a):
    done = sum(int(o[2].sum()) for o in run_a["outs"])
    goals = sum(int((o[3] != 0).sum()) for o in run_a["outs"])
    assert done > 0 and goals > 0, (done, goals)
    for cls in ("light", "heavy", "pair", "multi"):
        assert sum(c[cls] for c in run_a["classes"]) > 0, cls


@pytest.mark.parametrize("pre_steps", range(6))
def test_exact_resume_at_every_phase(run_a, pre_steps):
    n = run_a["n"]
    b = BatchedSoccerSim(n, config=CFG, seed=12345)
    b.reset(2, seed=777)
    for _ in range(pre_steps):  # another step counter and cache parity than A's
        b.step(torch.rand((n, 4, 3), device="cuda") * 2 - 1)
    b.load_state_dict(run_a["d"])
    assert b.stats() == run_a["stats0"]
    for t, (act, want) in enumerate(zip(run_a["acts"], run_a["outs"])):
        b.step(act)
        for x, y in zip(outputs(b), want):
            assert torch.equal(x, y), (pre_steps, t)
    assert torch.equal(b.save_states(), run_a["final"])
    sa, sb = dict(run_a["stats"]), b.stats()
    assert sa.pop("episode_return_sum") == pytest.approx(sb.pop("episode_return_sum"), rel=1e-6)
    assert sa == sb
    b.close()


def test_state_dict_checks_and_vecenv():
    v = TorchSoccerVecEnv(256, config=CFG, seed=1)
    v.reset({"use_full_random_positions": True}, seed=2)
    for _ in range(10):
        v.step(torch.rand((256, 4, 3), device="cuda") * 2 - 1)
    d = v.state_dict()
    assert set(d) >= {"format", "num_envs", "global_env_offset", "config", "states", "obs", "stats"}
    w = TorchSoccerVecEnv(256, config=CFG, seed=5)
    w.load_state_dict(d)
    assert torch.equal(w.sim.save_states(), v.sim.save_states()) and torch.equal(w.sim.obs, v.sim.obs)
    act = torch.rand((256, 4, 3), device="cuda") * 2 - 1
    assert all(torch.equal(x, y) for x, y in zip(v.step(act), w.step(act)))
    for other in (BatchedSoccerSim(128, config=CFG), BatchedSoccerSim(256, config=CFG, global_env_offset=256),
                  BatchedSoccerSim(256, config={**CFG, "simulation": {"max_steps": 61}})):
        with pytest.raises(ValueError):
            other.load_state_dict(d)
    with pytest.raises(ValueError):
        w.load_state_dict({**d, "format": "something else"})


def test_resharding_reproduces_the_whole_handle():
    n, h = 4096, 2048
    whole = staggered_sim(n, seed=13)
    d = whole.state_dict()
    halves = [BatchedSoccerSim(h, config=CFG, seed=99 + k, global_env_offset=k * h) for k in range(2)]
    for k, s in enumerate(halves):
        s.load_states(None, d["states"][k * h:(k + 1) * h])
        s.obs.copy_(d["obs"][k * h:(k + 1) * h])
    g = torch.Generator(device="cuda").manual_seed(3)
    resets = 0
    for t in range(130):
        act = torch.rand((n, 4, 3), generator=g, device="cuda") * 2 - 1
        whole.step(act)
        for k, s in enumerate(halves):
            s.step(act[k * h:(k + 1) * h].contiguous())
        for x, parts in zip(outputs(whole), zip(*[outputs(s) for s in halves])):
            assert torch.equal(x, torch.cat(parts)), t
        resets += int(whole.done.sum())
    assert resets > 0  # spawns after truncation, keyed by the global env index


def test_clone_envs():
    n = 4096
    sim, twin = staggered_sim(n, seed=17), staggered_sim(n, seed=17)
    inject_some(sim, [3], shift=40.0)
    inject_some(twin, [3], shift=40.0)
    rng = np.random.default_rng(0)
    dst = rng.choice(n, 600, replace=False)
    src = np.concatenate([[3], rng.choice(dst[:300], 299), rng.choice(n, 300)])  # repeats, overlaps dst
    assert len(set(src)) < len(src) and len(set(src) & set(dst)) > 0
    sim.clone_envs(src, dst)
    # the injected source clones with its flag: same record bytes, same picture
    assert torch.equal(sim.save_states([int(dst[0])]), twin.save_states([3]))
    assert torch.equal(sim.render([int(dst[0])], 84, 84), twin.render([3], 84, 84))
    assert torch.equal(sim.obs[dst], twin.obs[src])
    others = np.setdiff1d(np.arange(n), dst)
    dst_t, src_t, oth_t = (torch.from_numpy(x).cuda() for x in (dst, src, others))
    g = torch.Generator(device="cuda").manual_seed(4)
    ended = torch.zeros(len(dst), dtype=torch.bool, device="cuda")
    compared = 0
    for t in range(80):
        act = torch.rand((n, 4, 3), generator=g, device="cuda") * 2 - 1
        act_sim = act.clone()
        act_sim[dst_t] = act[src_t]
        sim.step(act_sim)
        twin.step(act)
        so, to = outputs(sim), outputs(twin)
        for x, y in zip(so, to):
            assert torch.equal(x[oth_t], y[oth_t]), t
        end_now = (so[2][dst_t] != 0) | (so[3][dst_t] != 0) | (to[2][src_t] != 0) | (to[3][src_t] != 0)
        ended |= end_now
        live = ~ended
        for x, y in zip(so, to):
            assert torch.equal(x[dst_t][live], y[src_t][live]), t
        compared += int(live.sum())
    assert compared > 600 * 20 and bool(ended.any())
    # clone_envs through CUDA tensors: pairs with an index out of range are skipped, without a device fault
    sim.clone_envs(torch.tensor([1, 2], device="cuda"), torch.tensor([2, 1], device="cuda"))
    before, obs = sim.save_states(), sim.obs.clone()
    sim.clone_envs(torch.tensor([1, n, 2, -1], device="cuda"), torch.tensor([5, 6, n, 7], device="cuda"))
    after = sim.save_states()
    assert torch.equal(after[5], before[1]) and torch.equal(sim.obs[5], obs[1])
    keep = [i for i in range(n) if i != 5]
    assert torch.equal(after[keep], before[keep]) and torch.equal(sim.obs[keep], obs[keep])
    sim.clone_envs(torch.tensor([n, -1], device="cuda"), torch.tensor([0, n], device="cuda"))  # no valid pair
    assert torch.equal(sim.save_states(), after) and torch.equal(sim.obs[keep], obs[keep])
    torch.cuda.synchronize()
    with pytest.raises(ValueError):
        sim.clone_envs([1, 2], [3, 3])


def test_saving_changes_nothing():
    n = 1024
    a, b = BatchedSoccerSim(n, config=CFG, seed=5), BatchedSoccerSim(n, config=CFG, seed=5)
    a.reset(2, seed=9); b.reset(2, seed=9)
    g = torch.Generator(device="cuda").manual_seed(1)
    out = torch.empty((n, B), dtype=torch.uint8, device="cuda")
    for t in range(150):
        act = torch.rand((n, 4, 3), generator=g, device="cuda") * 2.4 - 1.2
        a.step(act)
        b.save_states(out=out)
        b.save_states([0, 5, n - 1])
        b.step(act)
        for x, y in zip(outputs(a), outputs(b)):
            assert torch.equal(x, y), t
    sa, sb = a.stats(), b.stats()
    assert sa.pop("episode_return_sum") == pytest.approx(sb.pop("episode_return_sum"), rel=1e-6)
    assert sa == sb and sa["episodes"] > 0
    assert torch.equal(a.save_states(), b.save_states())


def test_index_handling():
    n = 300
    sim = staggered_sim(n, seed=4, steps=20)
    full = sim.save_states()
    dev = torch.tensor([3, n, -5, 1 << 40, 4], device="cuda")
    out = sim.save_states(dev)
    assert torch.equal(out[0], full[3]) and torch.equal(out[4], full[4]) and not out[1:4].any()
    other = staggered_sim(n, seed=8, steps=20).save_states()
    obs = sim.obs.clone()
    sim.load_states(torch.tensor([n, -1, 1 << 40], device="cuda"), other[:3])
    assert torch.equal(sim.save_states(), full) and torch.equal(sim.obs, obs)
    sim.load_states(torch.tensor([n, 7, -1], device="cuda"), other[:3])  # only the entry in range is installed
    now = sim.save_states()
    assert torch.equal(now[7], other[1]) and torch.equal(now[:7], full[:7]) and torch.equal(now[8:], full[8:])
    sim.load_states(None, full)
    for bad in ([0, n], [-1], [[1, 2]]):
        with pytest.raises(ValueError):
            sim.save_states(bad)
        with pytest.raises(ValueError):
            sim.load_states(bad, full[:len(np.ravel(bad))])
    with pytest.raises(ValueError):
        sim.load_states([4, 4], full[:2])
    with pytest.raises(ValueError):
        sim.load_states(None, torch.cat([full, full[:1]]))
    assert sim.save_states([]).shape == (0, B)
    sim.load_states([], full[:0])
    assert torch.equal(sim.save_states(), full)
    # misaligned slices: as input and as output
    raw = torch.zeros(n * B + 8, dtype=torch.uint8, device="cuda")
    mis = raw[8:].view(n, B)
    assert mis.data_ptr() % 16 == 8
    sim.save_states(out=mis)
    assert torch.equal(mis, full)
    sim.load_states(None, other)
    sim.load_states(list(range(n)), mis)
    assert torch.equal(sim.save_states(), full)
    sim.load_states([2, 1], full[[2, 1]].cpu())  # host tensors are moved to the device
    assert torch.equal(sim.save_states(), full)


def test_graph_capture_of_a_rewind_loop():
    n, k = 2048, 4
    sim, twin = staggered_sim(n, seed=6, steps=30), staggered_sim(n, seed=6, steps=30)
    start = sim.save_states()
    sim.load_states(None, start)  # the eager call that allocates what a load needs
    snap = torch.empty((n, B), dtype=torch.uint8, device="cuda")
    obs = [torch.empty_like(sim.obs) for _ in range(k)]
    act = torch.rand((k, n, 4, 3), device="cuda") * 2 - 1
    g = torch.cuda.CUDAGraph()
    torch.cuda.synchronize()
    with torch.cuda.graph(g):
        sim.save_states(out=snap)
        for i in range(k):
            sim.step(act[i])
            obs[i].copy_(sim.obs)
        sim.load_states(None, snap)
    want = []
    for i in range(k):  # the eager run of the same steps
        twin.step(act[i])
        want.append(twin.obs.clone())
    for rep in range(2):
        g.replay()
        torch.cuda.synchronize()
        for i in range(k):
            assert torch.equal(obs[i], want[i]), (rep, i)
        assert torch.equal(sim.save_states(), start), rep  # rewound
    # a fresh handle: the first load cannot be captured and says so, without a fault
    fresh = BatchedSoccerSim(n, config=CFG, seed=1)
    g2 = torch.cuda.CUDAGraph()
    with pytest.raises(_capi.MsocError):
        with torch.cuda.graph(g2):
            fresh.load_states(None, snap)
    torch.cuda.synchronize()
    fresh.load_states(None, snap)
    fresh.step(act[0])
    torch.cuda.synchronize()


def test_numpy_path_matches_device_path():
    n, seed = 512, 6
    dev, host = BatchedSoccerSim(n, config=CFG, seed=seed), HostBufferSim(n, CFG, seed=seed)
    dev.reset(2, seed=3); host.reset(2, seed=3)
    rng = np.random.default_rng(0)
    for _ in range(25):
        act = rng.uniform(-1, 1, (n, 4, 3)).astype(np.float32)
        dev.step(torch.from_numpy(act).cuda()); host.step(act)
    arr = host.save_states(np.arange(n))
    assert arr.dtype == _capi.ENV_STATE_DTYPE and arr.shape == (n,)
    assert np.array_equal(arr.view(np.uint8).reshape(n, B), dev.save_states().cpu().numpy())
    assert np.array_equal(host.save_states([7, 3]), arr[[7, 3]])
    other = HostBufferSim(n, CFG, seed=99)
    other.load_states(np.arange(n), arr)
    assert np.array_equal(other.save_states(np.arange(n)).view(np.uint8), arr.view(np.uint8))
    dev2 = BatchedSoccerSim(n, config=CFG, seed=1)
    dev2.load_states(None, torch.from_numpy(arr.view(np.uint8).reshape(n, B)).cuda())
    assert np.array_equal(dev2.save_states().cpu().numpy(), arr.view(np.uint8).reshape(n, B))


CHECKED = r"""
import sys
sys.path.insert(0, %(root)r); sys.path.insert(0, %(root)r + "/tests")
import numpy as np, torch
import parity_util as P
from marl_soccer_b200 import _capi
from marl_soccer_b200.sim import BatchedSoccerSim
L = _capi.lib()
assert L.msoc_debug_errors() == 0
cfg = {**P.CONFIG, "simulation": {"max_steps": 23}}
rng = np.random.default_rng(0)
for n in (1, 31, 33, 129, 70001):
    a, b = BatchedSoccerSim(n, config=cfg, seed=n), BatchedSoccerSim(n, config=cfg, seed=n + 1)
    a.reset(2, seed=1)
    for t in range(30):
        a.step(torch.rand((n, 4, 3), device="cuda") * 2 - 1)
    st = a.get_states([0]); st[0].hist_valid = 0; st[0].pos[1][0] += 30.0; a.set_states([0], st)
    snap = a.save_states()
    a.load_states(None, snap)
    a.save_states(torch.tensor([0, n, -1, n - 1], device="cuda"))
    a.load_states(torch.tensor([n, n - 1, -1], device="cuda"), snap[:3] if n >= 3 else snap[[0, 0, 0]])
    m = min(n, 500)
    src, dst = rng.integers(0, n, m), rng.permutation(n)[:m]
    a.clone_envs(src, dst)
    b.load_state_dict(a.state_dict())
    for t in range(25):
        act = torch.rand((n, 4, 3), device="cuda") * 2 - 1
        a.step(act); b.step(act)
    assert torch.equal(a.save_states(), b.save_states()), n
    bits = L.msoc_debug_errors()
    assert bits == 0, (n, bin(bits))
    a.close(); b.close()
print("checked build clean")
"""


def test_checked_build_states():
    from marl_soccer_b200 import build
    env = dict(os.environ, MSOC_LIB=build.build_checked())
    r = subprocess.run([sys.executable, "-c", CHECKED % {"root": ROOT}], env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "checked build clean" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]
