"""The picture of an env.  `scene(poses)` turns the five poses into draw primitives in screen coordinates -- the y axis
flipped like the reference's drawing code (soccer_simulation/renderer.py:30-42, game/entities.py:37-57,86-88) -- and is
the definition of what an env looks like.

Two paths draw it.  Batches of envs are rasterised on the GPU where they live: `BatchedSoccerSim.render()` /
`TorchSoccerVecEnv.render()` (uint8 CUDA tensors) and `HostBufferSim.render()` / `SyncMultiAgentVecEnv.render()`
(NumPy), all through msoc_render (csrc/render_core.cuh turns each primitive of `scene()` into an exact test on the
pixel centre).  `SoccerEnv(render_mode="human").render()` copies ONE env's poses to the host (msoc_get_state) and
`PygameRenderer` draws the primitives when pygame is installed; nothing in this module touches the GPU."""
from __future__ import annotations

import math

W, H, MARGIN, GOAL_H, AGENT, BALL_R = 800, 600, 10, 150, 30, 10  # game/constants.py
FIELD_RGB, LINE_RGB, BLUE_RGB, RED_RGB, BALL_RGB, NOSE_RGB = (34, 139, 34), (255, 255, 255), (0, 0, 255), (255, 0, 0), (255, 255, 255), (255, 255, 0)


def to_screen(x: float, y: float) -> tuple[float, float]:
    """World (y up) -> screen (y down)."""
    return float(x), float(H - y)


def _rot(px: float, py: float, ang: float) -> tuple[float, float]:
    c, s = math.cos(ang), math.sin(ang)
    return px * c - py * s, px * s + py * c


def scene(poses: dict) -> list:
    """poses: {"agents": [((x, y), angle) x 4], "ball": (x, y)} (SoccerEnv._game.poses()).  Returns a list of primitives
    ("line", rgb, p, q, width) / ("circle", rgb, centre, radius, width) / ("rect", rgb, (x, y, w, h), width) /
    ("poly", rgb, [points]) in screen coordinates, back to front."""
    mid_x, mid_y = W / 2, H / 2
    prims = [
        ("rect", FIELD_RGB, (0, 0, W, H), 0),
        ("line", LINE_RGB, (mid_x, MARGIN), (mid_x, H - MARGIN), 2),
        ("circle", LINE_RGB, (mid_x, mid_y), 70, 2),
        ("rect", LINE_RGB, (MARGIN, mid_y - 150, 120, 300), 2),
        ("rect", LINE_RGB, (W - MARGIN - 120, mid_y - 150, 120, 300), 2),
        ("rect", LINE_RGB, (0, mid_y - GOAL_H / 2, MARGIN, GOAL_H), 0),
        ("rect", LINE_RGB, (W - MARGIN, mid_y - GOAL_H / 2, MARGIN, GOAL_H), 0),
    ]
    half = AGENT / 2
    for i, ((x, y), ang) in enumerate(poses["agents"]):
        body = [to_screen(x + dx, y + dy) for dx, dy in (_rot(sx * half, sy * half, ang) for sx, sy in ((-1, -1), (1, -1), (1, 1), (-1, 1)))]
        prims.append(("poly", BLUE_RGB if i < 2 else RED_RGB, body))
        nose = [to_screen(x + dx, y + dy) for dx, dy in (_rot(px, py, ang) for px, py in ((half, 0.0), (half / 2, -half / 2), (half / 2, half / 2)))]
        prims.append(("poly", NOSE_RGB, nose))
    bx, by = poses["ball"]
    prims.append(("circle", BALL_RGB, to_screen(bx, by), BALL_R, 0))
    return prims


class PygameRenderer:
    """Draws `scene(poses)` in a pygame window (render_mode="human", soccer_env.py:156-162).  Constructing it without
    pygame raises ImportError; SoccerEnv.render() then returns the poses only."""

    def __init__(self, window_title: str = "Soccer Simulation"):
        import pygame
        self._pg = pygame
        pygame.init()
        self.screen = pygame.display.set_mode((W, H))
        pygame.display.set_caption(window_title)
        self.clock = pygame.time.Clock()

    def draw(self, poses: dict) -> None:
        pg = self._pg
        for event in pg.event.get():
            if event.type == pg.QUIT:
                pg.display.quit()
                return
        for p in scene(poses):
            if p[0] == "line":
                pg.draw.line(self.screen, p[1], p[2], p[3], p[4])
            elif p[0] == "circle":
                pg.draw.circle(self.screen, p[1], p[2], p[3], p[4])
            elif p[0] == "rect":
                pg.draw.rect(self.screen, p[1], p[2], p[3])
            else:
                pg.draw.polygon(self.screen, p[1], p[2])
        pg.display.flip()
        self.clock.tick(60)

    def close(self) -> None:
        self._pg.display.quit()
        self._pg.quit()
