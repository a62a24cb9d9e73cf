"""msoc_render on the device: the kernel against the fp64 reference rasteriser (tests/render_ref.py) on every pixel that
is not ambiguous, rendering leaves the simulation bit-identical, injected states, index handling, graph capture behind
msoc_step, the NumPy path, and the checked build."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import parity_util as P
import render_ref as R
from marl_soccer_b200 import _capi
from marl_soccer_b200.host_api import HostBufferSim
from marl_soccer_b200.marl_vecenv import SyncMultiAgentVecEnv, TorchSoccerVecEnv
from marl_soccer_b200.sim import BatchedSoccerSim

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CFG = {**P.CONFIG, "simulation": {"max_steps": 60}}


def staggered_sim(n, seed=0, steps=90):
    """n envs after a pre-roll with random actions and auto-reset; env i is re-spawned at step i % 60, so the episode
    phases are spread over the whole episode."""
    sim = BatchedSoccerSim(n, config=CFG, seed=seed)
    sim.reset(2, seed=seed + 1)
    g = torch.Generator(device="cuda").manual_seed(seed)
    ar = torch.arange(n, device="cuda")
    for t in range(steps):
        sim.step(torch.rand((n, 4, 3), generator=g, device="cuda") * 2 - 1)
        if t < 60:
            sim.reset(2, mask=(ar % 60 == t))
    return sim


def poses(sim, idx):
    return [R.poses_of_state(S) for S in sim.get_states(np.asarray(idx, np.int64))]


def test_kernel_matches_reference():
    n = 4096
    sim = staggered_sim(n, seed=3)
    ps = poses(sim, np.arange(n))
    report = {}
    for (H, W), m in [((96, 128), n), ((84, 84), n), ((37, 53), n), ((600, 800), 64)]:
        imgs = sim.render(None if m == n else torch.arange(m, device="cuda"), H, W).cpu().numpy()
        amb = bad = bad_clear = 0
        for img, pose in zip(imgs, ps[:m]):
            a, b, c = R.compare(img, pose)
            amb, bad, bad_clear = amb + a, bad + b, bad_clear + c
        report[f"{H}x{W}"] = {"images": m, "ambiguous_pixels": amb, "mismatches": bad, "mismatches_not_ambiguous": bad_clear}
        print(f"render {H}x{W} on {m} envs: {amb} ambiguous pixels, {bad} mismatches, {bad_clear} outside the ambiguous set")
        assert bad_clear == 0, (H, W, report)
    P.record("render_vs_reference", report)
    sim.close()


def test_rendering_changes_nothing():
    n = 1024
    a, b = BatchedSoccerSim(n, config=CFG, seed=5), BatchedSoccerSim(n, config=CFG, seed=5)
    a.reset(2, seed=9); b.reset(2, seed=9)
    g = torch.Generator(device="cuda").manual_seed(1)
    L = _capi.lib()
    host_out = np.empty((n, 37, 53, 3), np.uint8)
    for t in range(200):
        act = torch.rand((n, 4, 3), generator=g, device="cuda") * 2.4 - 1.2
        oa = [x.clone() for x in a.step(act)] + [a.score.clone()]
        b.render(None, 84, 84)
        _capi.check(L.msoc_render_host(b._h, None, n, 37, 53, host_out.ctypes.data))
        ob = [x.clone() for x in b.step(act)] + [b.score.clone()]
        for x, y in zip(oa, ob):
            assert torch.equal(x, y), t
    # the counters are exact; the return sum is added up per warp and then with atomics, and which envs share a warp
    # of the contact kernel varies from run to run (its work lists are filled by atomics), rendering or not
    sa_, sb_ = a.stats(), b.stats()
    assert sa_.pop("episode_return_sum") == pytest.approx(sb_.pop("episode_return_sum"), rel=1e-6)
    assert sa_ == sb_ and sa_["episodes"] > 0
    sa, sb = a.get_states(np.arange(n)), b.get_states(np.arange(n))
    assert all(bytes(x) == bytes(y) for x, y in zip(sa, sb))


def test_injected_state_shows_before_the_next_step():
    sim = staggered_sim(64, seed=2, steps=10)
    S = sim.get_states([7])[0]
    S.hist_valid = 0
    S.pos[2][0], S.pos[2][1], S.ang[2] = 120.0, 480.0, 0.7
    S.pos[4][0], S.pos[4][1] = 700.0, 90.0
    sim.set_states([7], [S])
    img = sim.render([7], 600, 800).cpu().numpy()[0]
    pose = R.poses_of_state(sim.get_states([7])[0])
    assert pose["agents"][2] == ((120.0, 480.0), pytest.approx(0.7))
    assert tuple(img[600 - 480, 120]) in ((255, 0, 0), (255, 255, 0)) and tuple(img[600 - 90, 700]) == (255, 255, 255)
    assert R.compare(img, pose)[2] == 0


def test_index_handling():
    n = 300
    sim = staggered_sim(n, seed=4, steps=20)
    full = sim.render(None, 37, 53)
    assert full.shape == (n, 37, 53, 3) and full.dtype == torch.uint8 and full.is_cuda
    idx = [299, 5, 5, 0, 150, 299]
    assert torch.equal(sim.render(idx, 37, 53), full[idx])
    assert torch.equal(sim.render(np.array(idx), 37, 53), full[idx])
    assert torch.equal(sim.render(torch.tensor(idx, device="cuda"), 37, 53), full[idx])
    for bad in ([0, n], [-1], [[1, 2]]):
        with pytest.raises(ValueError):
            sim.render(bad, 37, 53)
    dev = torch.tensor([3, n, -5, 1 << 40, 4], device="cuda")
    out = sim.render(dev, 37, 53)
    assert torch.equal(out[0], full[3]) and torch.equal(out[4], full[4])
    assert not out[1:4].any()
    # sizes that are not multiples of 16 bytes per row or per image, the smallest, and sizes whose tiles end inside a
    # warp's 32 segments (8 x 8: 2 432-pixel tiles), over all envs so that every image lies beside other tiles' images
    ps = poses(sim, np.arange(n))
    for H, W in [(1, 1), (3, 5), (8, 8), (84, 84)]:
        imgs = sim.render(None, H, W).cpu().numpy()
        for k in range(n):
            assert R.compare(imgs[k], ps[k])[2] == 0, (H, W, k)
    img = sim.render([17, 18], 1, 4096).cpu().numpy()
    for k in (0, 1):
        assert R.compare(img[k], ps[17 + k])[2] == 0
    with pytest.raises(_capi.MsocError):
        sim.render([0], 4097, 8)
    vec = TorchSoccerVecEnv(8, config=CFG, seed=1)
    assert torch.equal(vec.render([1, 2], 37, 53), vec.sim.render([1, 2], 37, 53))


def test_graph_capture_of_step_and_render():
    n, k, size = 2048, 3, (84, 84)
    a, b = BatchedSoccerSim(n, config=CFG, seed=8), BatchedSoccerSim(n, config=CFG, seed=8)
    a.reset(2, seed=1); b.reset(2, seed=1)
    act = torch.zeros((n, 4, 3), device="cuda")
    outs = [torch.empty((n, *size, 3), dtype=torch.uint8, device="cuda") for _ in range(k)]
    g = torch.cuda.CUDAGraph()
    torch.cuda.synchronize()
    with torch.cuda.graph(g):
        for i in range(k):
            a.step(act)
            a.render(None, *size, out=outs[i])
    gen = torch.Generator(device="cuda").manual_seed(2)
    for rep in range(3):
        act.copy_(torch.rand((n, 4, 3), generator=gen, device="cuda") * 2 - 1)
        g.replay()
        for i in range(k):
            b.step(act)
            assert torch.equal(outs[i], b.render(None, *size)), (rep, i)
    torch.cuda.synchronize()


def test_numpy_path_matches_device_path():
    n, seed = 512, 6
    dev, host = BatchedSoccerSim(n, config=CFG, seed=seed), HostBufferSim(n, CFG, seed=seed)
    vec = SyncMultiAgentVecEnv(None, num_envs=n, config=CFG, seed=seed)
    dev.reset(2, seed=3); host.reset(2, seed=3); vec.reset(options={"use_full_random_positions": True}, seed=3)
    rng = np.random.default_rng(0)
    for _ in range(15):
        act = rng.uniform(-1, 1, (n, 4, 3)).astype(np.float32)
        dev.step(torch.from_numpy(act).cuda()); host.step(act); vec.step(act)
    idx = [0, 511, 7, 7]
    for H, W in [(96, 128), (37, 53)]:
        want = dev.render(idx, H, W).cpu().numpy()
        assert np.array_equal(host.render(idx, H, W), want)
        assert np.array_equal(vec.render(idx, H, W), want)
    assert np.array_equal(host.render(None, 8, 8), dev.render(None, 8, 8).cpu().numpy())
    assert vec.render().shape == (1, 600, 800, 3)
    with pytest.raises(_capi.MsocError):
        host.render([n], 8, 8)


CHECKED = r"""
import sys
sys.path.insert(0, %(root)r); sys.path.insert(0, %(root)r + "/tests")
import numpy as np, torch
import parity_util as P
from marl_soccer_b200 import _capi
from marl_soccer_b200.sim import BatchedSoccerSim
from marl_soccer_b200.host_api import HostBufferSim
L = _capi.lib()
assert L.msoc_debug_errors() == 0
cfg = {**P.CONFIG, "simulation": {"max_steps": 23}}
for n in (1, 33, 1000):
    sim = BatchedSoccerSim(n, config=cfg, seed=n)
    sim.reset(2, seed=1)
    for t in range(30):
        sim.step(torch.rand((n, 4, 3), device="cuda") * 2 - 1)
    for H, W in ((1, 1), (3, 5), (37, 53), (84, 84), (600, 800), (2, 4096)):
        sim.render(None, H, W)
        sim.render([n - 1, 0, 0], H, W)
        sim.render(torch.tensor([0, n, -1, n - 1], device="cuda"), H, W)
    st = sim.get_states([0]); st[0].hist_valid = 0; st[0].pos[1][0] += 30.0; sim.set_states([0], st)
    sim.render(None, 37, 53)
    bits = L.msoc_debug_errors()
    assert bits == 0, (n, bin(bits))
    sim.close()
hs = HostBufferSim(100, cfg, seed=3)
hs.render([99, 0, 5], 37, 53); hs.render(None, 1, 1)
assert L.msoc_debug_errors() == 0
print("checked build clean")
"""


def test_checked_build_render():
    from marl_soccer_b200 import build
    env = dict(os.environ, MSOC_LIB=build.build_checked())
    r = subprocess.run([sys.executable, "-c", CHECKED % {"root": ROOT}], env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "checked build clean" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]
