"""TEST INFRASTRUCTURE: fp64 reference rasteriser of `renderer.scene(poses)`, the picture msoc_render draws.

Every primitive of the scene is an exact test on the pixel centre sx = (c + 0.5) 800 / W, sy = (r + 0.5) 600 / H:
  rect, width 0      x <= sx <= x + w and y <= sy <= y + h
  rect, width k      inside the rect and not strictly inside the rect inset by k
  line, width k      within k / 2 of the segment across it, between its end points along it
  circle, width 0    d <= r;  width k: r - k <= d <= r
  poly (convex)      on the inner side of every edge
The last primitive that covers a pixel gives its colour.  A pixel is ambiguous when its centre lies within EPS of the
boundary of any primitive (a superset is marked: near one edge of a half-plane set and within EPS of all the others);
the kernel computes in fp32 and may differ from this fp64 rasteriser there, and only there."""
from __future__ import annotations

import functools

import numpy as np

from marl_soccer_b200 import renderer

EPS = 1e-3
SW, SH = float(renderer.W), float(renderer.H)


def poses_of_state(S) -> dict:
    """The poses renderer.scene() takes, from an msoc_env_state (what SoccerEnv._game.poses() builds)."""
    return {"agents": [((float(S.pos[i][0]), float(S.pos[i][1])), float(S.ang[i])) for i in range(4)],
            "ball": (float(S.pos[4][0]), float(S.pos[4][1]))}


def _bounds(p):
    """Screen-unit bounding box (x0, x1, y0, y1) of a primitive."""
    kind = p[0]
    if kind == "rect":
        x, y, w, h = p[2]
        return x, x + w, y, y + h
    if kind == "line":
        (x0, y0), (x1, y1), k = p[2], p[3], p[4]
        return min(x0, x1) - k, max(x0, x1) + k, min(y0, y1) - k, max(y0, y1) + k
    if kind == "circle":
        (cx, cy), r = p[2], p[3]
        return cx - r, cx + r, cy - r, cy + r
    xs, ys = [q[0] for q in p[2]], [q[1] for q in p[2]]
    return min(xs), max(xs), min(ys), max(ys)


def _window(p, H, W):
    x0, x1, y0, y1 = _bounds(p)
    c0 = max(int(np.floor(x0 * W / SW - 0.5)) - 1, 0)
    c1 = min(int(np.ceil(x1 * W / SW - 0.5)) + 1, W - 1)
    r0 = max(int(np.floor(y0 * H / SH - 0.5)) - 1, 0)
    r1 = min(int(np.ceil(y1 * H / SH - 0.5)) + 1, H - 1)
    return r0, r1, c0, c1


def _halfplanes(gs):
    """gs: values g <= 0 inside.  Returns (inside, strictly inside, near the boundary)."""
    inside = np.logical_and.reduce([g <= 0 for g in gs])
    strict = np.logical_and.reduce([g < 0 for g in gs])
    near = np.logical_or.reduce([np.abs(g) <= EPS for g in gs]) & np.logical_and.reduce([g <= EPS for g in gs])
    return inside, strict, near


def _rect_g(x, y, w, h, X, Y):
    return [x - X, X - (x + w), y - Y, Y - (y + h)]


def _eval(p, X, Y):
    """(cover, ambiguous) of primitive p at the pixel centres X, Y."""
    kind = p[0]
    if kind == "rect":
        (x, y, w, h), k = p[2], p[3]
        cover, _, amb = _halfplanes(_rect_g(x, y, w, h, X, Y))
        if k:
            _, strict, amb_i = _halfplanes(_rect_g(x + k, y + k, w - 2 * k, h - 2 * k, X, Y))
            cover, amb = cover & ~strict, amb | amb_i
        return cover, amb
    if kind == "line":
        (x0, y0), (x1, y1), k = p[2], p[3], p[4]
        L = np.hypot(x1 - x0, y1 - y0)
        tx, ty = (x1 - x0) / L, (y1 - y0) / L
        along = (X - x0) * tx + (Y - y0) * ty
        across = -(X - x0) * ty + (Y - y0) * tx
        cover, _, amb = _halfplanes([-along, along - L, across - k / 2, -across - k / 2])
        return cover, amb
    if kind == "circle":
        (cx, cy), r, k = p[2], p[3], p[4]
        d = np.hypot(X - cx, Y - cy)
        if k == 0:
            return d <= r, np.abs(d - r) <= EPS
        return (d >= r - k) & (d <= r), (np.abs(d - r) <= EPS) | (np.abs(d - (r - k)) <= EPS)
    pts = [(float(a), float(b)) for a, b in p[2]]
    mx, my = sum(q[0] for q in pts) / len(pts), sum(q[1] for q in pts) / len(pts)
    gs = []
    for (ax, ay), (bx, by) in zip(pts, pts[1:] + pts[:1]):
        nx, ny = -(by - ay), bx - ax
        L = np.hypot(nx, ny)
        nx, ny = nx / L, ny / L
        if nx * (mx - ax) + ny * (my - ay) < 0:
            nx, ny = -nx, -ny
        gs.append(-(nx * (X - ax) + ny * (Y - ay)))
    cover, _, amb = _halfplanes(gs)
    return cover, amb


def _draw(prims, img, amb, H, W):
    for p in prims:
        r0, r1, c0, c1 = _window(p, H, W)
        if r0 > r1 or c0 > c1:
            continue
        X = (np.arange(c0, c1 + 1, dtype=np.float64) + 0.5) * SW / W
        Y = (np.arange(r0, r1 + 1, dtype=np.float64) + 0.5) * SH / H
        X, Y = np.meshgrid(X, Y)
        cover, near = _eval(p, X, Y)
        img[r0:r1 + 1, c0:c1 + 1][cover] = p[1]
        amb[r0:r1 + 1, c0:c1 + 1] |= near


@functools.lru_cache(maxsize=1)
def _static_count() -> int:
    """Number of leading primitives of scene() that do not depend on the poses (the field and its lines)."""
    a = renderer.scene({"agents": [((100.0, 100.0), 0.0)] * 4, "ball": (300.0, 300.0)})
    b = renderer.scene({"agents": [((500.0, 400.0), 1.0)] * 4, "ball": (600.0, 100.0)})
    n = 0
    while n < min(len(a), len(b)) and a[n] == b[n]:
        n += 1
    return n


@functools.lru_cache(maxsize=16)
def _background(H: int, W: int, statics: tuple):
    img = np.zeros((H, W, 3), np.uint8)
    amb = np.zeros((H, W), bool)
    _draw(list(statics), img, amb, H, W)
    img.setflags(write=False)
    amb.setflags(write=False)
    return img, amb


def rasterise(poses: dict, H: int, W: int):
    """(image (H, W, 3) uint8, ambiguous (H, W) bool) of scene(poses)."""
    prims = renderer.scene(poses)
    k = _static_count()
    bg, bg_amb = _background(H, W, tuple(prims[:k]))
    img, amb = bg.copy(), bg_amb.copy()
    _draw(prims[k:], img, amb, H, W)
    return img, amb


def compare(image: np.ndarray, poses: dict):
    """(ambiguous pixels, mismatching pixels, mismatching pixels that are not ambiguous) of one rendered image."""
    H, W = image.shape[:2]
    ref, amb = rasterise(poses, H, W)
    bad = np.any(image != ref, axis=-1)
    return int(amb.sum()), int(bad.sum()), int((bad & ~amb).sum())
