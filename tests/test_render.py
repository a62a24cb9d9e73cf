"""Rendering without a GPU: facts about the fp64 reference rasteriser (tests/render_ref.py, built from
renderer.scene()), the render kernel's own code compiled for the host (tests/hostsim/render_host.cu, render_core.cuh)
against that reference on every pixel that is not ambiguous, and argument checks of the C-ABI entry points."""
import ctypes as C
import math

import numpy as np
import pytest

import parity_util as P
import render_host_lib as RH
import render_ref as R
from hostsim_lib import HostSim
from marl_soccer_b200 import _capi, build, renderer

SIZES = [(600, 800), (96, 128), (84, 84), (37, 53), (1, 1)]
FACT_SIZES = [(600, 800), (96, 128), (84, 84)]


def poses(agents, ball):
    return {"agents": [((float(x), float(y)), float(a)) for x, y, a in agents], "ball": (float(ball[0]), float(ball[1]))}


SPREAD = poses([(150, 450, 0.0), (300, 120, math.pi / 2), (520, 470, 0.3), (650, 150, -2.0)], (250, 300))


def pixel_at(img, x, y):
    """The pixel whose area holds the world point (x, y) (y up)."""
    H, W = img.shape[:2]
    return tuple(int(v) for v in img[min(int((R.SH - y) * H / R.SH), H - 1), min(int(x * W / R.SW), W - 1)])


@pytest.mark.parametrize("H,W", FACT_SIZES)
def test_reference_ball_and_agent_centres(H, W):
    img, _ = R.rasterise(SPREAD, H, W)
    assert pixel_at(img, 250, 300) == renderer.BALL_RGB
    assert pixel_at(img, 150, 450) == renderer.BLUE_RGB and pixel_at(img, 300, 120) == renderer.BLUE_RGB
    assert pixel_at(img, 520, 470) == renderer.RED_RGB and pixel_at(img, 650, 150) == renderer.RED_RGB


@pytest.mark.parametrize("H,W", [(600, 800), (300, 400), (96, 128)])
def test_reference_noses_point_along_the_heading(H, W):
    """Angle 0 points to +x, angle pi/2 up the screen (world +y): the nose pixels of each agent lie ahead of it."""
    img, _ = R.rasterise(SPREAD, H, W)
    rows, cols = np.nonzero(np.all(img == renderer.NOSE_RGB, axis=-1))
    wx, wy = (cols + 0.5) * R.SW / W, R.SH - (rows + 0.5) * R.SH / H
    for (x, y), ang in SPREAD["agents"]:
        mine = np.hypot(wx - x, wy - y) < 20
        assert mine.sum() >= 1
        dx, dy = wx[mine].mean() - x, wy[mine].mean() - y
        assert abs(math.remainder(math.atan2(dy, dx) - ang, 2 * math.pi)) < 0.5
        assert 7.0 < math.hypot(dx, dy) < 13.0
    if H == 600:
        assert pixel_at(img, 150 + 12, 450) == renderer.NOSE_RGB and pixel_at(img, 150 - 12, 450) == renderer.BLUE_RGB
        assert pixel_at(img, 300, 120 + 12) == renderer.NOSE_RGB and pixel_at(img, 300, 120 - 12) == renderer.BLUE_RGB


def test_reference_flips_the_y_axis():
    img, _ = R.rasterise(poses([(200, 60, 0.0), (600, 540, 0.0), (700, 300, 0.0), (700, 400, 0.0)], (100, 500)), 600, 800)
    # world y = 60 is near the bottom of the image, y = 540 near the top
    assert tuple(img[600 - 60, 200]) == renderer.BLUE_RGB and tuple(img[600 - 540, 600]) == renderer.BLUE_RGB
    assert tuple(img[60, 200]) == renderer.FIELD_RGB and tuple(img[100, 100]) == renderer.BALL_RGB


def test_reference_field_lines():
    img, amb = R.rasterise(SPREAD, 600, 800)
    white, green = renderer.LINE_RGB, renderer.FIELD_RGB
    assert tuple(img[100, 400]) == white and tuple(img[100, 399]) == white and tuple(img[100, 402]) == green
    assert tuple(img[5, 400]) == green  # the centre line stops 10 units from the edge
    assert tuple(img[300, 469]) == white and tuple(img[300, 330]) == white and tuple(img[300, 466]) == green  # ring 68..70
    assert tuple(img[300, 5]) == white and tuple(img[300, 795]) == white  # goals
    assert tuple(img[200, 5]) == green  # beside the goal
    assert tuple(img[151, 60]) == white and tuple(img[300, 11]) == white and tuple(img[300, 60]) == green  # penalty box
    assert tuple(img[450, 700]) == green  # field
    # native size: every pixel centre is at least 0.5 units from the boundary of a field line
    lines = renderer.scene(SPREAD)[:R._static_count()]
    assert len(lines) == 7 and R._background(600, 800, tuple(lines))[1].sum() == 0


def test_reference_draw_order():
    # agent_2 (red) drawn over agent_1 (blue) where they overlap; the ball over an agent
    img, _ = R.rasterise(poses([(100, 100, 0.0), (400, 200, 0.0), (410, 200, 0.0), (600, 450, 0.0)], (600, 450)), 600, 800)
    assert pixel_at(img, 396, 200) == renderer.RED_RGB
    assert pixel_at(img, 390, 200) == renderer.BLUE_RGB
    assert pixel_at(img, 600, 450) == renderer.BALL_RGB and pixel_at(img, 600, 450 + 12) == renderer.RED_RGB
    img, _ = R.rasterise(poses([(100, 100, 0.0), (400, 200, 0.0), (388, 200, 0.0), (600, 450, 0.0)], (50, 50)), 600, 800)
    assert pixel_at(img, 402, 200) == renderer.NOSE_RGB  # agent_1's nose shows through nothing drawn later


def harness_states():
    """256 states: host-harness rollouts with random actions (rotated agents, contacts, corner spawns, auto-resets),
    then 64 of them moved partly outside the field by injection."""
    cfg = {**P.CONFIG, "simulation": {"max_steps": 29}}
    sim = HostSim(256, cfg, seed=5)
    sim.reset(2, seed=3)
    rng = np.random.default_rng(11)
    contacts = 0
    for _ in range(40):
        sim.step(rng.uniform(-1.0, 1.0, (256, 4, 3)).astype(np.float32))
        contacts += int(sim.last()[0].sum())
    assert contacts > 0
    for i in range(192, 256):
        S = sim.get_state(i)
        S.hist_valid = 0
        k = i % 5
        S.pos[k][0] = float(rng.choice([-8.0, 3.0, 796.0, 805.0]))
        S.pos[k][1] = float(rng.uniform(-8.0, 608.0))
        S.pos[(k + 1) % 5][1] = float(rng.choice([-6.0, 4.0, 597.0, 606.0]))
        S.ang[k % 4] = float(rng.uniform(-math.pi, math.pi))
        sim.set_state(i, S)
    states = [sim.get_state(i) for i in range(256)]
    return states, [R.poses_of_state(S) for S in states]


@pytest.fixture(scope="module")
def harness():
    return harness_states()


@pytest.mark.parametrize("H,W", SIZES)
def test_host_harness_matches_reference(harness, H, W):
    states, ps = harness
    imgs = RH.render(states, None, H, W)
    assert imgs.shape == (256, H, W, 3)
    total_amb = total_bad = 0
    for img, pose in zip(imgs, ps):
        amb, bad, bad_clear = R.compare(img, pose)
        assert bad_clear == 0
        total_amb += amb
        total_bad += bad
    # some index lists: reversed, with duplicates
    idx = np.array([255, 3, 3, 200, 0], np.int64)
    sub = RH.render(states, idx, H, W)
    assert np.array_equal(sub, imgs[idx])


def test_host_harness_out_of_range_index_is_zero(harness):
    states, _ = harness
    imgs = RH.render(states, np.array([1, 256, -1, 2], np.int64), 37, 53)
    assert not imgs[1].any() and not imgs[2].any()
    ref = RH.render(states, np.array([1, 2], np.int64), 37, 53)
    assert np.array_equal(imgs[0], ref[0]) and np.array_equal(imgs[3], ref[1])


def test_render_entry_points_reject_bad_arguments_without_a_device():
    L = C.CDLL(build.build())
    _capi.declare(L)
    out = (C.c_uint8 * 64)()
    assert L.msoc_render(None, None, 1, 4, 4, out, None) == -1
    assert L.msoc_render_host(None, None, 1, 4, 4, out) == -1
    # arguments are checked before the handle is used: a stand-in handle is never dereferenced here
    stand_in = (C.c_char * 8)()
    fake = C.c_void_p(C.addressof(stand_in))
    for n, h, w in [(-1, 4, 4), (1, 0, 4), (1, 4, 0), (1, 4097, 4), (1, 4, 4097)]:
        assert L.msoc_render(fake, None, n, h, w, out, None) == -1, (n, h, w)
        assert L.msoc_render_host(fake, None, n, h, w, out) == -1, (n, h, w)
    assert b"4096" in L.msoc_last_error()
    assert L.msoc_render(fake, None, 0, 4, 4, out, None) == 0  # n = 0 is a no-op
    assert L.msoc_render_host(fake, None, 0, 4, 4, out) == 0
