"""Synthetic input: the reference simulator's lidar and motion model, restated for the bench.

    lidar scan     slamrs/simulator/src/sim.rs:134-159  (one ray per beam, nearest segment hit,
                   `valid` = hit closer than scanner_range, else distance = range)
    ray/segment    slamrs/simulator/src/scene/ray.rs:55-83, 164-172
    motion model   slamrs/simulator/src/sim.rs:214-220
    odometry       slamrs/simulator/src/sim.rs:104-122 (wheel travel accumulated per tick)

f32 arithmetic like the reference; numpy's float32 cos/sin may differ from the platform libm by
an ulp, which only perturbs the synthetic scan, not the filter under test.
"""
from __future__ import annotations

import numpy as np

from .slam import Observation, Odometry

f32 = np.float32


def rect_segments(x, y, w, h):
    """Scene::add_rect, scene/ray.rs:124-149."""
    return [[x, y, x + w, y], [x + w, y, x + w, y + h], [x + w, y + h, x, y + h], [x, y + h, x, y]]


def reference_scene(scale: float = 1.0) -> np.ndarray:
    """The scene of slamrs/config/grid_slam.yaml:72-76, scaled about the origin."""
    seg = (rect_segments(-1.0, -1.0, 2.0, 2.0) + rect_segments(-0.1, -0.4, 0.5, 0.1) +
           rect_segments(-0.6, 0.4, 0.2, 0.5) + [[-0.6, -0.4, 0.2, 0.4]])
    return (np.array(seg, np.float64) * scale).astype(np.float32)


def scene_map(segments, config) -> np.ndarray:
    """A probability map of the scene for a grid of `config` (a GridMapSlamConfig): 0.9 on every cell a segment
    crosses, 0.5 (unknown) elsewhere; flat f64, index row * grid_h + column, the layout of estimated_likelihood().
    A segment is sampled every quarter cell, both endpoints included; a sample marks the cell it falls in
    (Map::world_to_grid and is_valid, map.rs:60-69). Deterministic, so tests and benchmarks get a map without a
    SLAM run."""
    from .slam import grid_cells
    gw, gh = grid_cells(config.width, config.resolution), grid_cells(config.height, config.resolution)
    res, px, py = f32(config.resolution), f32(config.position[0]), f32(config.position[1])
    out = np.full(gw * gh, 0.5, np.float64)
    for x1, y1, x2, y2 in np.asarray(segments, np.float32).reshape(-1, 4):
        length = float(np.hypot(float(x2) - float(x1), float(y2) - float(y1)))
        k = max(1, int(np.ceil(4.0 * length / float(res))))
        t = np.linspace(0.0, 1.0, k + 1, dtype=np.float32)
        gx = (x1 + (x2 - x1) * t - px) / res
        gy = (y1 + (y2 - y1) * t - py) / res
        ok = (gx >= 0) & (gy >= 0) & (gx < gw) & (gy < gh)
        out[gy[ok].astype(np.int64) * gh + gx[ok].astype(np.int64)] = 0.9
    return out


def scan(segments: np.ndarray, pose, n_beams: int, scanner_range: float) -> Observation:
    px, py, pt = f32(pose[0]), f32(pose[1]), f32(pose[2])
    deg = np.arange(n_beams, dtype=np.float32) * f32(360.0 / n_beams)
    ang = deg * (f32(np.pi) / f32(180.0))                     # f32::to_radians
    d = ang + pt
    dx, dy = np.cos(d, dtype=np.float32), np.sin(d, dtype=np.float32)
    x1, y1, x2, y2 = (segments[:, k][None, :] for k in range(4))
    x3, y3 = px, py
    x4, y4 = (px + dx)[:, None], (py + dy)[:, None]
    with np.errstate(divide="ignore", invalid="ignore"):
        denom = (x1 - x2) * (y3 - y4) - (y1 - y2) * (x3 - x4)
        t = ((x1 - x3) * (y3 - y4) - (y1 - y3) * (x3 - x4)) / denom
        u = -((x1 - x2) * (y1 - y3) - (y1 - y2) * (x1 - x3)) / denom
    ok = (denom != 0) & (t >= 0) & (t <= 1) & (u > 0)
    u = np.where(ok, u, np.inf).astype(np.float32)
    best = u.min(axis=1)
    have = np.isfinite(best)                                   # rays that hit nothing are dropped (sim.rs:138)
    rng = f32(scanner_range)
    valid = best < rng
    dist = np.where(valid, best, rng).astype(np.float32)
    return Observation(0, angle=ang[have].astype(np.float64), distance=dist[have].astype(np.float64), valid=valid[have])


class Simulator:
    """Fixed-timestep differential-drive robot with a 360-degree lidar (sim.rs:96-212)."""

    def __init__(self, segments, n_beams=360, scanner_range=1.0, wheel_base=0.1, update_period=1.0, dt=1.0 / 30.0):
        self.segments = np.ascontiguousarray(segments, np.float32)
        self.n_beams, self.scanner_range = n_beams, f32(scanner_range)
        self.wheel_base, self.update_period, self.dt = f32(wheel_base), f32(update_period), f32(dt)
        self.pose = [f32(0), f32(0), f32(0)]
        self.timer = f32(0)
        self.acc = [f32(0), f32(0)]
        self.counter = 0

    def _motion(self, sl, sr):
        sbar = (sr + sl) / f32(2.0)
        self.pose[2] = f32(self.pose[2] + (sr - sl) / self.wheel_base)
        self.pose[0] = f32(self.pose[0] + sbar * np.cos(self.pose[2], dtype=np.float32))
        self.pose[1] = f32(self.pose[1] + sbar * np.sin(self.pose[2], dtype=np.float32))

    def next_scan(self, speed_left: float, speed_right: float):
        """Ticks at dt until the scanner fires; returns (Observation, Odometry)."""
        vl, vr = f32(speed_left), f32(speed_right)
        while True:
            self._motion(vl * self.dt, vr * self.dt)
            self.acc[0] = f32(self.acc[0] + vl * self.dt)
            self.acc[1] = f32(self.acc[1] + vr * self.dt)
            self.timer = f32(self.timer + self.dt)
            if self.timer > self.update_period:
                self.timer = f32(self.timer - self.update_period)
                odo = Odometry.new(float(self.acc[0]), float(self.acc[1]), float(self.wheel_base))
                self.acc = [f32(0), f32(0)]
                obs = scan(self.segments, self.pose, self.n_beams, self.scanner_range)
                obs.id = self.counter
                self.counter += 1
                return obs, odo
