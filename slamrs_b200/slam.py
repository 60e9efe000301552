"""Host-side mirror of the reference's grid SLAM interface, on top of the C ABI.

Names, argument meaning and error behaviour follow the Rust items they stand in for:

    Pose, Measurement, Observation, Odometry   slamrs/common/src/robot.rs:9-184
    GridMapSlamConfig, GridMapSlam             slamrs/slam/src/grid/slam.rs:13-97
    GridData                                   slamrs/slam/src/grid/map.rs:181-264

so that a test written against `GridMapSlam::{new, update, estimated_pose,
estimated_likelihood, map_position}` reads the same here. All computation happens in
libslamrs_gpu.so on the GPU; nothing in this module computes the filter on the CPU.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import Iterable, Optional, Sequence

import numpy as np

from . import _lib

# ln(0.3/0.7), ln(0.9/(1-0.9)): the two non-zero inverse-sensor-model increments (map.rs:154-156)
L_FREE = float(np.log(np.float64(0.30) / (np.float64(1.0) - np.float64(0.30))))
L_OCC = float(np.log(np.float64(0.9) / (np.float64(1.0) - np.float64(0.9))))


@dataclass
class Pose:
    """robot.rs:9-18 (f32 fields)."""
    x: float = 0.0
    y: float = 0.0
    theta: float = 0.0

    def xy(self):
        return (self.x, self.y)


@dataclass
class Measurement:
    """robot.rs:82-94."""
    angle: float
    distance: float
    strength: float = 1.0
    valid: bool = True


class Observation:
    """robot.rs:51-54. Stored column-wise (f64 angle/distance, bool valid) for cheap hand-off."""

    def __init__(self, id: int = 0, measurements: Optional[Iterable[Measurement]] = None, *,
                 angle=None, distance=None, valid=None):
        self.id = id
        if measurements is not None:
            ms = list(measurements)
            self.angle = np.array([m.angle for m in ms], np.float64)
            self.distance = np.array([m.distance for m in ms], np.float64)
            self.valid = np.array([m.valid for m in ms], np.bool_)
        else:
            self.angle = np.ascontiguousarray(angle if angle is not None else [], np.float64)
            self.distance = np.ascontiguousarray(distance if distance is not None else [], np.float64)
            self.valid = np.ascontiguousarray(valid if valid is not None else [], np.bool_)
        if not (self.angle.shape == self.distance.shape == self.valid.shape):
            raise ValueError("angle, distance and valid must have the same length")

    @property
    def measurements(self):
        return [Measurement(float(a), float(d), 1.0, bool(v)) for a, d, v in zip(self.angle, self.distance, self.valid)]

    def __len__(self):
        return int(self.angle.size)


@dataclass
class Odometry:
    """robot.rs:115-129. The two Normal distributions are derived inside the library exactly as
    Odometry::new does (robot.rs:132-150); only the three measured floats cross the boundary."""
    distance_left: float
    distance_right: float
    wheel_distance: float

    @staticmethod
    def new(distance_left: float, distance_right: float, wheel_distance: float) -> "Odometry":
        return Odometry(distance_left, distance_right, wheel_distance)


@dataclass
class GridMapSlamConfig:
    """slam.rs:18-25 -- the YAML block `config:` of a `!GridMapSlam` node (config/grid_slam.yaml:24-29)."""
    position: Sequence[float] = (-2.0, -2.0)
    width: float = 4.0
    height: float = 4.0
    resolution: float = 0.02
    n_particles: int = 10


@dataclass
class GridData:
    """map.rs:181-264: `size` in cells and a flat row-major `data` vector, index = row*size.y + column."""
    size: tuple
    data: np.ndarray

    def iter_cells(self):
        sy = self.size[1]
        for i, v in enumerate(self.data):
            yield (i // sy, i % sy), v  # (row, column), map.rs:206-214


@dataclass
class GpuPlacement:
    """What the YAML cannot carry: device, shard, RNG mode (see INTEGRATION.md)."""
    device: int = -1
    rank: int = 0
    world_size: int = 1
    nccl_id: Optional[bytes] = None
    seed: int = 0x5EED5A11
    rng_mode: int = _lib.RNG_SHARED_STREAM
    spare_slots: int = 0
    flags: int = 0
    resample_threshold: float = 0.0   # 0 = resample after every update (the reference); tau: only when N_eff < tau * N
    slot_cells: int = 0      # 0 = whole-grid slots; power of two >= 256 = windowed slots (see slamrs_gpu.h)


@dataclass
class ScanMatcher:
    """Scan-matching pose refinement of the SLAM step (slamrs_gpu_scan_match; not in the reference, off by default).
    Each sampled pose climbs, before the likelihood, to the pose whose beam endpoints lie nearest to occupied cells of
    its particle's own map: `radius` cells around each endpoint are searched (0..2), the climb tries steps of
    `step_xy` metres and `step_theta` radians, halves them `levels` - 1 times (1..8) and stops after `max_moves`
    accepted moves (1..1024). The defaults are what the quality measurement in DESIGN.md used."""
    radius: int = 1
    step_xy: float = 0.1
    step_theta: float = 0.05
    levels: int = 4
    max_moves: int = 32

    def to_struct(self):
        m = _lib.ScanMatch()
        m.struct_size = C.sizeof(_lib.ScanMatch)
        m.radius, m.levels, m.max_moves = int(self.radius), int(self.levels), int(self.max_moves)
        m.step_xy, m.step_theta = float(self.step_xy), float(self.step_theta)
        return m


def grid_cells(extent: float, resolution: float) -> int:
    """Map::new grid sizing (map.rs:28-31) as the library computes it."""
    out = C.c_uint32(0)
    _lib.check(_lib.load().slamrs_gpu_grid_cells(extent, resolution, C.byref(out)))
    return int(out.value)


def nccl_unique_id() -> bytes:
    buf = (C.c_uint8 * _lib.NCCL_ID_BYTES)()
    _lib.check(_lib.load().slamrs_gpu_nccl_unique_id(buf))
    return bytes(buf)


def _ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class GridMapSlam:
    """GridMapSlam (slam.rs:13-97) running on one B200 (or one shard of a multi-GPU filter)."""

    def __init__(self, config: GridMapSlamConfig, placement: Optional[GpuPlacement] = None):
        self._L = _lib.load()
        self._h = C.c_void_p()
        pl = placement or GpuPlacement()
        self.config = config
        self.placement = pl
        if config.n_particles <= 0:
            raise ValueError("Must have at least one particle")  # particle.rs:16 assert
        gw = grid_cells(config.width, config.resolution)
        gh = grid_cells(config.height, config.resolution)
        self._create(self._config_struct(config, pl, gw, gh))
        self.grid_w, self.grid_h = gw, gh
        self.n_particles = int(config.n_particles)
        self.n_local = self.n_particles // pl.world_size
        self.first = pl.rank * self.n_local

    def _create(self, cfg) -> None:
        _lib.check(self._L.slamrs_gpu_create(C.byref(cfg), C.byref(self._h)))

    @staticmethod
    def _config_struct(config: GridMapSlamConfig, pl: GpuPlacement, gw: int, gh: int):
        cfg = _lib.Config()
        cfg.struct_size = C.sizeof(_lib.Config)
        cfg.abi_version = _lib.ABI_VERSION
        cfg.pos_x, cfg.pos_y = float(config.position[0]), float(config.position[1])
        cfg.resolution = float(config.resolution)
        cfg.grid_w, cfg.grid_h = gw, gh
        cfg.n_particles = int(config.n_particles)
        cfg.seed = int(pl.seed)
        cfg.rng_mode = int(pl.rng_mode)
        cfg.device = int(pl.device)
        cfg.rank, cfg.world_size = int(pl.rank), int(pl.world_size)
        cfg.spare_slots = int(pl.spare_slots)
        cfg.flags = int(pl.flags)
        cfg.slot_cells = int(pl.slot_cells)
        cfg.resample_threshold = float(pl.resample_threshold)
        if pl.world_size > 1:
            if pl.nccl_id is None or len(pl.nccl_id) != _lib.NCCL_ID_BYTES:
                raise ValueError("world_size > 1 needs the 128-byte nccl_id shared by all ranks")
            C.memmove(cfg.nccl_id, pl.nccl_id, _lib.NCCL_ID_BYTES)
        return cfg

    @classmethod
    def new(cls, config: GridMapSlamConfig, placement: Optional[GpuPlacement] = None) -> "GridMapSlam":
        return cls(config, placement)

    # ------------------------------------------------------------------ lifecycle
    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self._L.slamrs_gpu_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # ------------------------------------------------------------------ the reference API
    @staticmethod
    def _scan_arrays(z: Observation):
        # `m.angle as f32`, `m.distance as f32` (map.rs:76-77, 121-122)
        return (np.ascontiguousarray(z.angle, np.float32), np.ascontiguousarray(z.distance, np.float32),
                np.ascontiguousarray(z.valid, np.uint8))

    def update(self, z: Observation, u: Odometry, z_draws: Optional[np.ndarray] = None,
               resample_u: Optional[float] = None) -> None:
        """GridMapSlam::update (slam.rs:46-75). `z_draws`/`resample_u` only in RNG_CALLER mode."""
        angle, dist, valid = self._scan_arrays(z)
        zd = None if z_draws is None else np.ascontiguousarray(z_draws, np.float64)
        if zd is not None and zd.size != 2 * self.n_particles:
            raise ValueError("z_draws must hold 2 * n_particles values")
        ru = None if resample_u is None else np.array([resample_u], np.float64)
        _lib.check(self._L.slamrs_gpu_update(self._h, _ptr(angle), _ptr(dist), _ptr(valid), angle.size,
                                             u.distance_left, u.distance_right, u.wheel_distance,
                                             _ptr(zd), _ptr(ru)), self._h)

    def estimated_pose(self) -> Pose:
        out = np.zeros(3, np.float32)
        _lib.check(self._L.slamrs_gpu_pose(self._h, _ptr(out)), self._h)
        return Pose(float(out[0]), float(out[1]), float(out[2]))

    def estimated_likelihood(self, out: Optional[np.ndarray] = None) -> GridData:
        if out is None:
            out = np.empty(self.grid_w * self.grid_h, np.float64)
        _lib.check(self._L.slamrs_gpu_map_probability(self._h, _ptr(out)), self._h)
        return GridData((self.grid_w, self.grid_h), out)

    def estimated_likelihood_async(self, out: Optional[np.ndarray]) -> None:
        """Pipelined estimated_likelihood(): queues the conversion behind the steps issued so far and the copy into
        `out` (flat f64, grid_w * grid_h, page-locked host memory) on the handle's copy stream, and returns; `out` holds
        the map after map_wait(). The next update() may be issued first: the copy overlaps it. Multi-GPU: every rank
        calls it, `out=None` on ranks that only take part."""
        if out is not None and (out.dtype != np.float64 or out.size < self.grid_w * self.grid_h):
            raise ValueError("out must be a flat float64 buffer of grid_w * grid_h cells")
        _lib.check(self._L.slamrs_gpu_map_probability_async(self._h, None if out is None else _ptr(out)), self._h)

    def map_wait(self) -> None:
        """Blocks until every pending estimated_likelihood_async() copy has landed in its buffer."""
        _lib.check(self._L.slamrs_gpu_map_wait(self._h), self._h)

    def skip_estimated_likelihood(self) -> None:
        """Multi-GPU: take part in the other ranks' estimated_likelihood() without receiving the map."""
        _lib.check(self._L.slamrs_gpu_map_probability(self._h, None), self._h)

    def skip_estimated_likelihood_window(self) -> None:
        """Multi-GPU: take part in the other ranks' estimated_likelihood_window() (extent + window) without the map."""
        self.map_extent()
        _lib.check(self._L.slamrs_gpu_map_window(self._h, _lib.MAP_F32, 0, 0, 0, 0, None), self._h)

    def map_extent(self):
        """(x0, y0, x1, y1): informed extent of the estimate's grid in cells; all zero for an empty map."""
        out = np.zeros(4, np.int32)
        _lib.check(self._L.slamrs_gpu_map_extent(self._h, _ptr(out)), self._h)
        return tuple(int(v) for v in out)

    def estimated_likelihood_window(self, window=None, fmt: int = _lib.MAP_F32, out: Optional[np.ndarray] = None) -> tuple:
        """((x0, y0, x1, y1), array[y1-y0, x1-x0]) of the estimate's map in f64 / f32 / u8; the default
        window is the informed extent -- every cell outside it is exactly 0.5. `out`: a flat buffer of
        the right dtype to fill (e.g. pinned host memory), at least window-sized."""
        x0, y0, x1, y1 = window if window is not None else self.map_extent()
        dt = {_lib.MAP_F64: np.float64, _lib.MAP_F32: np.float32, _lib.MAP_U8: np.uint8}[fmt]
        shape = (max(0, y1 - y0), max(0, x1 - x0))
        if out is not None:
            if out.dtype != dt or out.size < shape[0] * shape[1]:
                raise ValueError("out buffer has the wrong dtype or is too small")
            out = out.reshape(-1)[:shape[0] * shape[1]].reshape(shape)
        else:
            out = np.empty(shape, dt)
        if out.size:
            _lib.check(self._L.slamrs_gpu_map_window(self._h, fmt, x0, y0, x1, y1, _ptr(out)), self._h)
        return (x0, y0, x1, y1), out

    def number_of_effective_particles(self) -> float:
        """particle.rs:59-65 on the last update's normalised weights (before resampling)."""
        out = C.c_double(0.0)
        _lib.check(self._L.slamrs_gpu_effective_particles(self._h, C.byref(out)), self._h)
        return float(out.value)

    # ------------------------------------------------------------------ scan production on the device
    def sim_scan(self, segments, pose, n_beams: int, scanner_range: float) -> int:
        """The simulator's lidar evaluated on the device into the handle's scan buffers; returns the
        number of measurements. Follow with step_async()."""
        seg = np.ascontiguousarray(segments, np.float32).reshape(-1, 4)
        p = np.ascontiguousarray(pose, np.float32).reshape(3)
        n = C.c_uint32(0)
        _lib.check(self._L.slamrs_gpu_sim_scan(self._h, _ptr(seg), seg.shape[0], _ptr(p), n_beams, scanner_range,
                                               C.byref(n)), self._h)
        return int(n.value)

    def get_scan(self) -> Observation:
        n = C.c_uint32(0)
        _lib.check(self._L.slamrs_gpu_get_scan(self._h, None, None, None, 0, C.byref(n)), self._h)
        a = np.zeros(n.value, np.float32); d = np.zeros(n.value, np.float32); v = np.zeros(n.value, np.uint8)
        if n.value:
            _lib.check(self._L.slamrs_gpu_get_scan(self._h, _ptr(a), _ptr(d), _ptr(v), n.value, C.byref(n)), self._h)
        return Observation(0, angle=a.astype(np.float64), distance=d.astype(np.float64), valid=v.astype(bool))

    def map_position(self):
        return tuple(self.config.position)  # slam.rs:90-96: constant, answered from the config

    # ------------------------------------------------------------------ pipelined form
    def upload_scan(self, z: Observation) -> None:
        angle, dist, valid = self._scan_arrays(z)
        _lib.check(self._L.slamrs_gpu_upload_scan(self._h, _ptr(angle), _ptr(dist), _ptr(valid), angle.size), self._h)

    def step_async(self, u: Odometry, z_draws: Optional[np.ndarray] = None, resample_u: Optional[float] = None) -> None:
        zd = None if z_draws is None else np.ascontiguousarray(z_draws, np.float64)
        ru = None if resample_u is None else np.array([resample_u], np.float64)
        _lib.check(self._L.slamrs_gpu_step_async(self._h, u.distance_left, u.distance_right, u.wheel_distance,
                                                 _ptr(zd), _ptr(ru)), self._h)

    def set_scan_device(self, angle_ptr: int, dist_ptr: int, valid_ptr: int, n_beams: int, max_dist: float) -> None:
        """Step on an observation that already lives in device memory (raw device pointers). `max_dist` bounds
        |distance| over every beam (it sizes the ray kernel's window); +inf, NaN or <= 0 mean unknown and are exact for
        any scan. A bound that some beam exceeds can make the step fail with E_INTERNAL."""
        _lib.check(self._L.slamrs_gpu_set_scan_device(self._h, angle_ptr, dist_ptr, valid_ptr, n_beams, max_dist), self._h)

    def set_profiling(self, enabled: bool) -> None:
        _lib.check(self._L.slamrs_gpu_set_profiling(self._h, int(enabled)), self._h)

    def phase_ms(self):
        """(dict phase -> summed ms, steps covered) since the last call; synchronises."""
        ms = np.zeros(len(_lib.PHASES), np.float64); steps = C.c_uint64(0)
        _lib.check(self._L.slamrs_gpu_get_phase_ms(self._h, _ptr(ms), C.byref(steps)), self._h)
        return dict(zip(_lib.PHASES, ms.tolist())), int(steps.value)

    def step_history(self, first_step: int, count: int) -> np.ndarray:
        """count x {grids_copied, grids_pulled, distinct_sources, source_reads, particles_integrated,
        copy_bytes}."""
        out = np.zeros((count, _lib.HISTORY_VALUES), np.uint64)
        _lib.check(self._L.slamrs_gpu_get_step_history(self._h, first_step, count, _ptr(out)), self._h)
        return out

    def sync(self) -> None:
        _lib.check(self._L.slamrs_gpu_sync(self._h), self._h)

    @property
    def stream_ptr(self) -> int:
        return int(self._L.slamrs_gpu_stream(self._h) or 0)

    @property
    def launch_count(self) -> int:
        return int(self._L.slamrs_gpu_launch_count(self._h))

    # ------------------------------------------------------------------ scan matching (extension)
    def set_scan_matcher(self, matcher: Optional[ScanMatcher]) -> None:
        """Refine every sampled pose by scan matching from the next update on; None turns it off (the default).
        Multi-GPU: every rank sets the same matcher before the same update."""
        m = None if matcher is None else matcher.to_struct()
        _lib.check(self._L.slamrs_gpu_set_scan_match(self._h, None if m is None else C.byref(m)), self._h)

    def scan_match_stats(self) -> dict:
        """Of this rank's particles in the last update: moved (particles), moves (total), scored (poses, start poses
        included), capped (particles that stopped at max_moves). All zero after an update without the matcher."""
        out = np.zeros(4, np.uint64)
        _lib.check(self._L.slamrs_gpu_get_scan_match_stats(self._h, _ptr(out)), self._h)
        return dict(zip(("moved", "moves", "scored", "capped"), (int(v) for v in out)))

    # ------------------------------------------------------------------ introspection (tests / bench)
    def stats(self) -> dict:
        s = _lib.Stats()
        _lib.check(self._L.slamrs_gpu_get_stats(self._h, C.byref(s)), self._h)
        return {n: int(getattr(s, n)) for n, _ in _lib.Stats._fields_}

    def poses(self) -> np.ndarray:
        out = np.zeros((self.n_local, 3), np.float32)
        _lib.check(self._L.slamrs_gpu_get_poses(self._h, _ptr(out)), self._h)
        return out

    def slots(self):
        """(slot_of[n_local], spare[n_spare]): the resampler's slot table and spare list."""
        n = C.c_uint32(0)
        _lib.check(self._L.slamrs_gpu_get_slots(self._h, None, None, C.byref(n)), self._h)
        slot_of = np.zeros(self.n_local, np.int32); spare = np.zeros(int(n.value), np.int32)
        _lib.check(self._L.slamrs_gpu_get_slots(self._h, _ptr(slot_of), _ptr(spare) if spare.size else None, C.byref(n)), self._h)
        return slot_of, spare

    def extents(self, particle: int):
        """((x0, y0, x1, y1), shift, bands[n_bands, 2]): informed box, row rotation and per-band column ranges
        (x0, x1) of one particle's grid as the resampler sees them."""
        box = np.zeros(5, np.int32); n = C.c_uint32(0)
        _lib.check(self._L.slamrs_gpu_get_extents(self._h, particle, _ptr(box), None, C.byref(n)), self._h)
        raw = np.zeros(int(n.value), np.uint32)
        _lib.check(self._L.slamrs_gpu_get_extents(self._h, particle, _ptr(box), _ptr(raw), C.byref(n)), self._h)
        return tuple(int(v) for v in box[:4]), int(box[4]), np.column_stack([raw & 0xFFFF, raw >> 16]).astype(np.int64)

    def init_uniform(self, box) -> None:
        """Uniform start poses over box = (x0, y0, x1, y1) metres, heading in [-pi, pi), from the shared stream
        (global-localisation-style initialisation; README.md:45)."""
        b = np.ascontiguousarray(box, np.float32).reshape(4)
        _lib.check(self._L.slamrs_gpu_init_uniform(self._h, _ptr(b)), self._h)

    def set_poses(self, xyt) -> None:
        a = np.ascontiguousarray(xyt, np.float32).reshape(self.n_local, 3)
        _lib.check(self._L.slamrs_gpu_set_poses(self._h, _ptr(a)), self._h)

    def weights(self):
        norm = np.zeros(self.n_particles, np.float64); raw = np.zeros(self.n_particles, np.float64)
        _lib.check(self._L.slamrs_gpu_get_weights(self._h, _ptr(norm), _ptr(raw)), self._h)
        return norm, raw

    def resample_indices(self) -> np.ndarray:
        out = np.zeros(self.n_particles, np.uint32)
        _lib.check(self._L.slamrs_gpu_get_resample_indices(self._h, _ptr(out)), self._h)
        return out

    @property
    def max_particle(self) -> int:
        out = C.c_uint64(0)
        _lib.check(self._L.slamrs_gpu_get_max_particle(self._h, C.byref(out)), self._h)
        return int(out.value)

    def cells(self, particle: int) -> np.ndarray:
        out = np.zeros(self.grid_w * self.grid_h, np.uint32)
        _lib.check(self._L.slamrs_gpu_get_cells(self._h, particle, _ptr(out)), self._h)
        return out

    def set_cells(self, particle: int, cells) -> None:
        a = np.ascontiguousarray(cells, np.uint32).reshape(-1)
        assert a.size == self.grid_w * self.grid_h
        _lib.check(self._L.slamrs_gpu_set_cells(self._h, particle, _ptr(a)), self._h)

    def counts(self, particle: int):
        c = self.cells(particle)
        return (c & 0xFFFF).astype(np.uint16), (c >> 16).astype(np.uint16)

    def log_odds(self, particle: int) -> np.ndarray:
        out = np.zeros(self.grid_w * self.grid_h, np.float64)
        _lib.check(self._L.slamrs_gpu_get_log_odds(self._h, particle, _ptr(out)), self._h)
        return out


@dataclass
class SensorModel:
    """How a GridMapLocalizer scores a beam endpoint against its loaded map (slamrs_gpu_sensor_model).

    kind SENSOR_BEAM_ENDPOINT (the default, as every extension here defaults to the reference): Map::probability_of's
    factor (map.rs:130-141). It scores endpoints in unknown space or off the map best, so it cannot localise from a
    uniform start; it is there for parity with the SLAM step. Global localisation needs kind SENSOR_LIKELIHOOD_FIELD:
    log(z_hit * exp(-d^2 / (2 sigma^2)) + z_rand), d = distance to the nearest cell with p > occupied_above."""
    kind: int = _lib.SENSOR_BEAM_ENDPOINT
    sigma: float = 0.1            # metres
    z_rand: float = 0.05          # z_hit = 1 - z_rand
    occupied_above: float = 0.5

    @staticmethod
    def likelihood_field(sigma: float = 0.1, z_rand: float = 0.05, occupied_above: float = 0.5) -> "SensorModel":
        return SensorModel(_lib.SENSOR_LIKELIHOOD_FIELD, sigma, z_rand, occupied_above)

    def to_struct(self):
        m = _lib.SensorModel()
        m.struct_size = C.sizeof(_lib.SensorModel)
        m.kind, m.sigma, m.z_rand, m.occupied_above = int(self.kind), float(self.sigma), float(self.z_rand), float(self.occupied_above)
        return m


class GridMapLocalizer(GridMapSlam):
    """Monte Carlo localisation against a loaded occupancy map: GridMapSlam::update with the map held fixed and shared
    by every particle (no per-particle grids). `map_probability` is the grid_w * grid_h f64 probabilities, flat or
    2-D (index row * grid_h + column), or the GridData that GridMapSlam.estimated_likelihood() returns. Place the
    particles with init_uniform() or set_poses(), then update() and estimated_pose() as on a GridMapSlam; the grid
    read-outs (estimated_likelihood, cells, ...) raise. Runs on one GPU (placement.world_size must be 1)."""

    def __init__(self, config: GridMapSlamConfig, map_probability, model: Optional[SensorModel] = None,
                 placement: Optional[GpuPlacement] = None):
        data = map_probability.data if isinstance(map_probability, GridData) else map_probability
        self._map = np.ascontiguousarray(data, np.float64).reshape(-1)
        self.model = model or SensorModel()
        super().__init__(config, placement)

    def _create(self, cfg) -> None:
        if self._map.size != cfg.grid_w * cfg.grid_h:
            raise ValueError(f"map_probability holds {self._map.size} cells, the grid {cfg.grid_w * cfg.grid_h}")
        m = self.model.to_struct()
        _lib.check(self._L.slamrs_gpu_create_localizer(C.byref(cfg), C.byref(m), _ptr(self._map), C.byref(self._h)))

    def sensor_terms(self) -> np.ndarray:
        """The grid_w * grid_h f64 term table the device built from the map (index row * grid_h + column)."""
        out = np.zeros(self.grid_w * self.grid_h, np.float64)
        _lib.check(self._L.slamrs_gpu_get_sensor_terms(self._h, _ptr(out)), self._h)
        return out


# ---------------------------------------------------------------------- kernel-level hooks
def debug_raycast(x0, y0, x1, y1, grid_w, grid_h, extra=2, cap=None, device=0):
    x0, y0, x1, y1 = (np.ascontiguousarray(v, np.float32).reshape(-1) for v in (x0, y0, x1, y1))
    n = x0.size
    cap = int(cap or (grid_w + grid_h + 16))
    out = np.zeros((n, cap, 2), np.int32)
    cnt = np.zeros(n, np.uint32)
    _lib.check(_lib.load().slamrs_gpu_debug_raycast(device, _ptr(x0), _ptr(y0), _ptr(x1), _ptr(y1), n, grid_w, grid_h,
                                                    extra, _ptr(out), cap, _ptr(cnt)))
    return out, cnt


def debug_sincos(x, device=0):
    x = np.ascontiguousarray(x, np.float32).reshape(-1)
    s = np.zeros_like(x); c = np.zeros_like(x)
    _lib.check(_lib.load().slamrs_gpu_debug_sincos(device, _ptr(x), x.size, _ptr(s), _ptr(c)))
    return s, c


def debug_stream(seed, step, first, count, device=0):
    z = np.zeros(2 * count, np.float64); u = np.zeros(1, np.float64)
    _lib.check(_lib.load().slamrs_gpu_debug_stream(device, seed, step, first, count, _ptr(z), _ptr(u)))
    return z, float(u[0])


def debug_resample(raw_weights, u01: float, device=0, timing=False, tau=0.0):
    """normalize_weights + argmax + resample indices on the device for caller-supplied raw weights
    (the step's own k_weights / k_resample_indices) with the adaptive-resampling threshold tau
    (resample_threshold). Returns a dict: idx, max_particle, norm, cum, clamped, fold_rounds, fold_heads,
    fold_fallback, n_eff, do_resample, and the launch k_weights used: cluster (CTAs), threads (per CTA), chunk
    (elements per thread), regs (elements in registers, else the generic kernel) (+ us = (k_weights,
    k_resample_indices) with timing)."""
    w = np.ascontiguousarray(raw_weights, np.float64).reshape(-1)
    n = w.size
    idx = np.zeros(n, np.uint32); norm = np.zeros(n, np.float64); cum = np.zeros(n, np.float64)
    info = np.zeros(4, np.uint64); us = np.zeros(2, np.float32); mp = C.c_uint64(0)
    n_eff = C.c_double(0.0); do_resample = C.c_uint64(0); shape = np.zeros(4, np.uint64)
    _lib.check(_lib.load().slamrs_gpu_debug_resample_adaptive(
        device, _ptr(w), n, float(u01), float(tau), _ptr(idx), C.byref(mp), _ptr(norm), _ptr(cum), _ptr(info),
        _ptr(us) if timing else None, C.byref(n_eff), C.byref(do_resample), _ptr(shape)))
    out = dict(idx=idx, max_particle=int(mp.value), norm=norm, cum=cum, clamped=int(info[0]), fold_rounds=int(info[1]),
               fold_heads=int(info[2]), fold_fallback=int(info[3]), n_eff=float(n_eff.value),
               do_resample=bool(do_resample.value), cluster=int(shape[0]), threads=int(shape[1]), chunk=int(shape[2]),
               regs=bool(shape[3]))
    if timing:
        out["us"] = (float(us[0]), float(us[1]))
    return out
