"""The fused ray update's parked hits (k_ray_update_half), in lockstep with the CPU oracle. A 16-bit window cell counts
at most 31 occupied hits; the 32nd and later occupied hits of a cell in one scan, and every hit of a zero-length ray,
are parked per work item and added to the grid after the write-back. The lower half's parked hits on the start row
travel to the upper half, which owns that row. These tests fill both lists to and past the sizes they once had (60
start-row hits, 4 per ray) with crowded start rows, rays that emit five occupied cells, zero-length rays, clones and
saturating counters, on the fused kernel and, as the control, on the generic kernel. Each case computes on the host,
with the reference's walk, how many hits it parks, and shows from stats() that it ran the fused kernel and parked."""
import math

import numpy as np
import pytest

from oracle import oracle as O
from oracle.scan_match_oracle import ScanMatchOracle
from slamrs_b200 import GpuPlacement, GridMapSlam, GridMapSlamConfig, Observation, Odometry, _lib, grid_cells
from slamrs_b200.simulator import Simulator, reference_scene

from common import SEED, compare_step, install_cells, lockstep_following_device_weights

pytestmark = pytest.mark.gpu

f32 = np.float32
RAY_PACKED_MAX_BEAMS = 2047
PK_OCC_MAX = 31                 # occupied hits a 16-bit window cell holds
OLD_START_ROW_CAP = 60          # the start-row list the exchange record once had
OLD_SPILL_CAP = 4 * RAY_PACKED_MAX_BEAMS
FLAGS = {"fused": 0, "generic": _lib.FLAG_GENERIC_RAY_KERNEL}
CROWD_CFG = GridMapSlamConfig(position=(-6.4, -6.4), width=12.8, height=12.8, resolution=0.05, n_particles=4)
WIDE_CFG = GridMapSlamConfig(position=(-12.8, -12.8), width=25.6, height=25.6, resolution=0.05, n_particles=4)


# ------------------------------------------------------------------------------------------------ host model
def _half_window_cells(radius):
    """kernels_ray.cu ray_window_cells_upper_bound_half."""
    worst = 0
    for a in range(8):
        total = 0
        for dy in range(radius + 1):
            hw, cx = math.isqrt(radius * radius - dy * dy), 4096 + a
            total += ((cx + hw + 1 + 7) & ~7) - ((cx - hw) & ~7)
        worst = max(worst, total)
    return worst


def _fused_window(cfg, obs):
    maxd = float(np.max(np.abs(obs.distance.astype(f32))))
    radius = min(int(math.ceil(f32(maxd) / f32(cfg.resolution))) + 6, 150)
    return 2 * _half_window_cells(radius)


def _occupied_hits(cfg, pose, obs):
    """Per half (False: lower, True: upper) a dict cell -> occupied hits of one scan from `pose`, with the step's f32
    arithmetic (beam endpoint, world_to_grid, the reference's walk and sensor model)."""
    gw = grid_cells(cfg.width, cfg.resolution)
    gh = grid_cells(cfg.height, cfg.resolution)
    px0, py0, res = f32(cfg.position[0]), f32(cfg.position[1]), f32(cfg.resolution)
    x, y, th = (f32(v) for v in pose)
    sx, sy = f32((x - px0) / res), f32((y - py0) / res)
    ang, dist = obs.angle.astype(f32), obs.distance.astype(f32)
    a = (th + ang).astype(f32)
    s, c = O.libm_sincosf(a)
    gx = (((x + (c * dist).astype(f32)).astype(f32) - px0) / res).astype(f32)
    gy = (((y + (s * dist).astype(f32)).astype(f32) - py0) / res).astype(f32)
    out = {False: {}, True: {}}
    for b in range(len(ang)):
        upper = not gy[b] < sy
        md = f32(dist[b] / res)
        for cx, cy in O.ray_cells(float(sx), float(sy), float(gx[b]), float(gy[b]), gw, gh):
            dx = f32(sx - f32(f32(cx) + f32(0.5)))
            dy = f32(sy - f32(f32(cy) + f32(0.5)))
            d = np.sqrt(f32(f32(dx * dx) + f32(dy * dy)), dtype=f32)
            if O.inverse_sensor_model(float(d), float(md), bool(obs.valid[b])) == 2:
                key = (int(cx), int(cy))
                out[upper][key] = out[upper].get(key, 0) + 1
    return out, int(np.floor(sy))


def _parked(cfg, pose, obs):
    """(lower half's parked start-row hits, parked hits per half) of one still step from an empty grid."""
    occ, cy0 = _occupied_hits(cfg, pose, obs)
    over = {u: {k: n - PK_OCC_MAX for k, n in occ[u].items() if n > PK_OCC_MAX} for u in occ}
    start_row = sum(n for (cx, cy), n in over[False].items() if cy == cy0)
    return start_row, {u: sum(over[u].values()) for u in over}, occ


# ------------------------------------------------------------------------------------------------ lockstep
class _OddsFromDevice:
    """The oracle with the device's log-odds: a saturated counter's log-odds keep the unbounded sum in the oracle
    (DESIGN.md), so only counters are compared there."""

    def __init__(self, f, gpu):
        self._f, self._gpu = f, gpu

    def __getattr__(self, name):
        return getattr(self._f, name)

    def odds(self, p):
        return self._gpu.log_odds(p)


def _still(cfg, observations, poses, flags, cells=None, saturated=False):
    """Lockstep with every particle held where it was placed (odometry 0, caller draws z = 0). `cells`: particle ->
    packed counters installed on both sides first. Returns stats() per step."""
    n = cfg.n_particles
    odo = Odometry.new(0.0, 0.0, 0.1)
    z = np.zeros(2 * n)
    out = []
    gpu = GridMapSlam(cfg, GpuPlacement(seed=SEED, rng_mode=_lib.RNG_CALLER, flags=flags))
    osl = ScanMatchOracle(cfg.position, cfg.width, cfg.height, cfg.resolution, n, True)   # (set_counts)
    try:
        gpu.set_poses(poses)
        osl.set_poses(poses)
        for p, c in (cells or {}).items():
            install_cells(gpu, osl, p, c)
        for step, obs in enumerate(observations):
            u = O.resample_uniform(SEED, step)
            ang = obs.angle.astype(f32).astype(np.float64)
            dist = obs.distance.astype(f32).astype(np.float64)
            assert osl.update(ang, dist, obs.valid.astype(np.uint8), f32(0.0), f32(0.0), f32(0.1), z, u) == 0
            gpu.update(obs, odo, z_draws=z, resample_u=u)
            compare_step(gpu, _OddsFromDevice(osl, gpu) if saturated else osl, check_map=not saturated)
            out.append((gpu.stats(), osl.indices().copy()))
    finally:
        gpu.close()
        osl.close()
    return out


def _obs(angle, dist, valid):
    return Observation(0, angle=np.asarray(angle, np.float64), distance=np.asarray(dist, np.float64),
                       valid=np.asarray(valid, bool))


def _check_ran(stats, obs, cfg, flags):
    """The fused kernel ran and parked hits; or the generic kernel ran."""
    if flags == "fused":
        assert stats["window_cells"] == _fused_window(cfg, obs), stats
        assert stats["spilled_cells"] > 0, stats
    else:
        assert stats["window_cells"] != _fused_window(cfg, obs), stats


# ------------------------------------------------------------------------------------------------ 1. recorded scene
def test_recorded_scene_near_a_wall():
    """configs[1]'s scene at 64 particles (test_gpu_scan_match.quality_run): at step 16 the robot is 2 mm from a
    wall and every particle's lower half parks about a hundred start-row hits. Lockstep through step 22 on the fused
    and the generic kernel; the grids of every particle are compared at steps 16 to 21."""
    cfg = GridMapSlamConfig(position=(-12.8, -12.8), width=25.6, height=25.6, resolution=0.05, n_particles=64)
    sim = Simulator(reference_scene(5.0), n_beams=360, scanner_range=6.0, wheel_base=0.1)
    scans = [sim.next_scan(0.08, 0.10) for _ in range(23)]
    everyone = list(range(cfg.n_particles))
    _, _, stats = lockstep_following_device_weights(
        O, cfg, scans, lambda step, idx, gpu: everyone if 16 <= step <= 21 else [], check_map=False,
        flags=[FLAGS["fused"], FLAGS["generic"]])
    assert stats[16][0]["window_cells"] == _fused_window(cfg, scans[16][0])
    assert stats[16][0]["spilled_cells"] > 0


# ------------------------------------------------------------------------------------------------ 2. crowded start row
def _crowd_pose(cfg, cy0, up):
    """Start cell (128, cy0), half a cell across; near the top of the cell for the downward fan (it stays on the start
    row), near the bottom for the mirrored one."""
    res = cfg.resolution
    fy = 0.95 if not up else 0.05
    return (f32(cfg.position[0] + 128.5 * res), f32(cfg.position[1] + (cy0 + fy) * res), f32(0.0))


def _crowd_scan(cfg, n_a, n_b, up):
    """n_a beams of 0.2 m and n_b of 0.21 m, heading 0.01 rad below (above: `up`) the +x axis, all valid: their
    occupied runs overlap on the start row."""
    sgn = 1.0 if up else -1.0
    ang = np.full(n_a + n_b, sgn * 0.01)
    dist = np.concatenate([np.full(n_a, 4 * cfg.resolution), np.full(n_b, 4.2 * cfg.resolution)])
    return _obs(ang, dist, np.ones(n_a + n_b, bool))


def _crowd_counts(cfg, target, cy0, up):
    """(parked, n_a, n_b) with the fewest beams whose parked hits (the lower half's on the start row; mirrored: the
    upper half's) equal `target`, or the nearest above when none does. One beam of each kind is walked; n identical
    beams put n times its hits on each of its cells."""
    pose = _crowd_pose(cfg, cy0, up)
    half = {k: _occupied_hits(cfg, pose, _crowd_scan(cfg, *k, up))[0][up] for k in ((1, 0), (0, 1))}
    cells = set(half[(1, 0)]) | set(half[(0, 1)])
    if not up:
        cells = {c for c in cells if c[1] == cy0}
    best = None
    for n_a in range(0, 120):
        for n_b in range(0, 120):
            got = sum(max(0, n_a * half[(1, 0)].get(c, 0) + n_b * half[(0, 1)].get(c, 0) - PK_OCC_MAX) for c in cells)
            if got >= target and (best is None or (got, n_a + n_b) < (best[0], best[1] + best[2])):
                best = (got, n_a, n_b)
    return best


@pytest.mark.parametrize("flags", ["fused", "generic"])
@pytest.mark.parametrize("cy0", [128, 131, 0, 1, 254, 255])
@pytest.mark.parametrize("target", [59, 60, 61])
@pytest.mark.parametrize("up", [False, True], ids=["lower", "mirrored"])
def test_crowded_start_row(flags, cy0, target, up):
    cfg = CROWD_CFG
    got, n_a, n_b = _crowd_counts(cfg, target, cy0, up)
    assert got == target, (got, n_a, n_b)
    obs = _crowd_scan(cfg, n_a, n_b, up)
    pose = _crowd_pose(cfg, cy0, up)
    start_row, per_half, _ = _parked(cfg, pose, obs)
    if up:
        assert start_row == 0 and per_half[False] == 0 and per_half[True] == target
    else:
        assert per_half[True] == 0 and start_row == per_half[False] == target
    assert (start_row > OLD_START_ROW_CAP) == (target > OLD_START_ROW_CAP and not up)
    out = _still(cfg, [obs, obs], np.array([pose] * cfg.n_particles, f32), FLAGS[flags])
    _check_ran(out[0][0], obs, cfg, flags)


@pytest.mark.parametrize("flags", ["fused", "generic"])
@pytest.mark.parametrize("cy0", [128, 131, 0, 255])
def test_a_thousand_start_row_hits(flags, cy0):
    cfg = CROWD_CFG
    pose = _crowd_pose(cfg, cy0, False)
    obs = _crowd_scan(cfg, 31 + 500, 0, False)   # two occupied start-row cells per beam
    start_row, per_half, _ = _parked(cfg, pose, obs)
    assert 990 <= start_row == per_half[False] <= 1010, start_row
    out = _still(cfg, [obs, obs], np.array([pose] * cfg.n_particles, f32), FLAGS[flags])
    _check_ran(out[0][0], obs, cfg, flags)


# ------------------------------------------------------------------------------------------------ 3. the total list
FIVE_START = (200.8050537, 200.9636688)   # cell units: this start, heading and distance emit five occupied cells
FIVE_ANGLE, FIVE_DIST = 0.9457754, 1.4466372


def _five_pose(cfg, mirror):
    """The start point of the five-cell ray in WIDE_CFG's cells; `mirror`: reflected about the cell's mid-row."""
    res = cfg.resolution
    fy = FIVE_START[1] - 200.0
    y = 200.0 + (1.0 - fy if mirror else fy)
    return (f32(cfg.position[0] + FIVE_START[0] * res), f32(cfg.position[1] + y * res), f32(0.0))


def _five_beam(cfg, pose, down, need=5):
    """A heading near the recorded one (mirrored: downward) whose ray from `pose` emits `need` occupied cells."""
    res = cfg.resolution
    for k in range(0, 4000):
        for sgn in (1, -1):
            a = FIVE_ANGLE + sgn * k * 1e-5
            a = -a if down else a
            obs = _obs([a], [FIVE_DIST * res], [True])
            occ, _ = _occupied_hits(cfg, pose, obs)
            if sum(occ[not down].values()) >= need and not occ[down]:
                return a
    raise AssertionError(f"no {need}-cell heading near the recorded one")


def _total_scan(cfg, kind):
    """2,047 beams: five-cell rays up, down or split, or mixed with zero-length rays. Returns (pose, obs)."""
    res = cfg.resolution
    down = kind == "down"
    pose = _five_pose(cfg, mirror=down)
    n = RAY_PACKED_MAX_BEAMS
    if kind == "split":
        a_up = _five_beam(cfg, pose, False)
        a_dn = _five_beam(cfg, pose, True, need=4)
        ang = np.where(np.arange(n) % 2 == 0, a_up, a_dn)
        dist = np.full(n, FIVE_DIST * res)
    else:
        ang = np.full(n, _five_beam(cfg, pose, down))
        dist = np.full(n, FIVE_DIST * res)
        if kind == "zero_length":
            dist[1000:] = 1e-9                     # px + cos(a) 1e-9 rounds back to px: dx = dy = 0
    return pose, _obs(ang, dist, np.ones(n, bool))


@pytest.mark.parametrize("flags", ["fused", "generic"])
@pytest.mark.parametrize("kind", ["up", "down", "split", "zero_length"])
def test_total_list(flags, kind):
    cfg = WIDE_CFG
    pose, obs = _total_scan(cfg, kind)
    _, per_half, occ = _parked(cfg, pose, obs)
    zero = int(np.count_nonzero(obs.distance < 1e-6))
    parked = {u: per_half[u] for u in per_half}
    parked[True] += 3 * zero                       # a zero-length ray parks all three hits (upper half: y_inc = 0)
    if kind == "up":
        assert parked[True] > OLD_SPILL_CAP and parked[False] == 0, parked
    if kind == "down":
        assert parked[False] > OLD_SPILL_CAP and parked[True] == 0, parked
    if kind == "split":
        assert parked[False] > 0 and parked[True] > 0, parked
    if kind == "zero_length":
        assert parked[True] > 3 * zero > 0, parked
    assert max(parked.values()) <= 7 * RAY_PACKED_MAX_BEAMS
    out = _still(cfg, [obs, obs], np.array([pose] * cfg.n_particles, f32), FLAGS[flags])
    _check_ran(out[0][0], obs, cfg, flags)


# ------------------------------------------------------------------------------------------------ 4. clones
def _disc_cells(cfg, pose, packed, radius_cells=20):
    """Packed counters `packed` in every cell within `radius_cells` of the start cell, zero elsewhere."""
    gw = grid_cells(cfg.width, cfg.resolution)
    cx = int((pose[0] - f32(cfg.position[0])) / f32(cfg.resolution))
    cy = int((pose[1] - f32(cfg.position[1])) / f32(cfg.resolution))
    c = np.zeros(gw * gw, np.uint32)
    yy, xx = np.mgrid[0:gw, 0:gw]
    c[((xx - cx) ** 2 + (yy - cy) ** 2 <= radius_cells ** 2).reshape(-1)] = packed
    return c


@pytest.mark.parametrize("flags", ["fused", "generic"])
@pytest.mark.parametrize("case", ["crowded_131", "crowded_128", "total_down", "total_split"])
def test_clones_park_into_their_own_slot(flags, case):
    """Every particle resamples particle 0: three fused clones and the owner integrate the crowded scan. The clones'
    parked hits land in their own slots after their write-back; the root's owner waits for them. Particle 0's grid
    holds occupied cells (an endpoint likelihood of 0.9 p + 0.1, about 1); the others hold free cells where the beams
    end, which makes their weights negligible, and the clones' write-back must clear them."""
    if case.startswith("crowded"):
        cfg = CROWD_CFG
        cy0 = int(case.split("_")[1])
        pose = _crowd_pose(cfg, cy0, False)
        obs = _crowd_scan(cfg, 31 + 100, 0, False)
        assert _parked(cfg, pose, obs)[0] > OLD_START_ROW_CAP
    else:
        cfg = WIDE_CFG
        pose, obs = _total_scan(cfg, case.split("_")[1])
    out = _still(cfg, [obs, obs], np.array([pose] * cfg.n_particles, f32), FLAGS[flags],
                 cells={p: _disc_cells(cfg, pose, (5 << 16) if p == 0 else 5) for p in range(cfg.n_particles)})
    idx = out[0][1]
    assert np.all(idx == 0), idx                   # one source for every survivor: clones
    _check_ran(out[0][0], obs, cfg, flags)


# ------------------------------------------------------------------------------------------------ 5. saturation
@pytest.mark.parametrize("flags", ["fused", "generic"])
@pytest.mark.parametrize("side", ["below", "at", "above"])
def test_parked_start_row_hits_saturate(flags, side):
    """Start-row cells preloaded near 65,535 occupied hits on every particle: the lower half's parked hits reach the
    limit exactly, stop one short, or pass it."""
    cfg = CROWD_CFG
    cy0 = 131
    pose = _crowd_pose(cfg, cy0, False)
    obs = _crowd_scan(cfg, 31 + 100, 0, False)
    start_row, _, occ = _parked(cfg, pose, obs)
    assert start_row > OLD_START_ROW_CAP
    gw = grid_cells(cfg.width, cfg.resolution)
    hits = {k: n for k, n in occ[False].items() if k[1] == cy0}
    slack = {"below": -1, "at": 0, "above": 1}[side]
    c = np.zeros(gw * gw, np.uint32)
    for (cx, cy), n in hits.items():
        c[cy * gw + cx] = np.uint32(65535 - n + slack) << np.uint32(16)
    out = _still(cfg, [obs], np.array([pose] * cfg.n_particles, f32), FLAGS[flags],
                 cells={p: c for p in range(cfg.n_particles)}, saturated=True)
    stats = out[0][0]
    assert (stats["counter_saturated"] > 0) == (side == "above"), stats
    _check_ran(stats, obs, cfg, flags)
