"""Scan shapes and distances the simulator never produces, in lockstep with the CPU oracle: the beam counts at which
the ray kernels change (sort, packed and fused kernels, the 32-bit generic kernel), non-finite, zero, negative,
subnormal and huge distances and the classifier's band edges, zero-length rays, device-resident scans, the
localiser's beam windows and partial warps, and the likelihood-field distance transform at edge maps and sizes.
Every test also shows that it reached the branch it is about, from what the library reports."""
import math

import numpy as np
import pytest
import torch
from scipy import ndimage

from oracle import loc_oracle as LO
from slamrs_b200 import (GpuPlacement, GridMapLocalizer, GridMapSlam, GridMapSlamConfig, Observation, Odometry,
                         SensorModel, _lib, grid_cells)
from slamrs_b200.simulator import reference_scene, scene_map

from common import SEED, WEIGHT_RTOL, at_scale_config, compare_step, lockstep, make_scans, oracle_slam, oracle_step

pytestmark = pytest.mark.gpu

RAY_PACKED_MAX_BEAMS = 2047                    # kernels_ray.cu: the packed window's 11-bit free field
RAY_SPILL_CAP = 7 * RAY_PACKED_MAX_BEAMS       # parked hits per work item of the fused ray update
SORT_MAX_BEAMS = 2048                          # k_sort_beams
LOC_WIN = 1024                                 # k_loc_step: scan beams per window
FLAGS = {"default": 0, "generic": _lib.FLAG_GENERIC_RAY_KERNEL}
MODELS = {"beam": SensorModel(), "field": SensorModel.likelihood_field(sigma=0.1, z_rand=0.05)}
f32 = np.float32


def preset(n=8):
    """The shipped preset's 200^2 grid at 2 cm (1 m lidar: scans mix valid and invalid beams)."""
    return GridMapSlamConfig(position=(-2.0, -2.0), width=4.0, height=4.0, resolution=0.02, n_particles=n)


def _rel(a, b):
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-300)))


def _obs(angle, dist, valid):
    return Observation(0, angle=np.asarray(angle, np.float64), distance=np.asarray(dist, np.float64),
                       valid=np.asarray(valid, bool))


class _NanAsOne:
    """A filter whose weights() read NaN as 1 (compare_step's relative errors are NaN for NaN)."""

    def __init__(self, f):
        self._f = f

    def __getattr__(self, name):
        return getattr(self._f, name)

    def weights(self):
        return tuple(np.where(np.isnan(w), 1.0, w) for w in self._f.weights())


class _OddsFromDevice(_NanAsOne):
    """The oracle, with the device's log-odds in place of its own (for saturated counters, see _compare)."""

    def __init__(self, f, gpu):
        super().__init__(f)
        self._gpu = gpu

    def odds(self, p):
        return self._gpu.log_odds(p)


def _compare(gpu, osl, saturated=False):
    """compare_step, where a scan with thousands of valid beams may drive every raw weight to 0: the reference's
    normalised weights are then 0/0 = NaN, and the device's must be NaN in the same places. `saturated`: the step
    saturates hit counters, which the oracle saturates too, but its log-odds keep the unbounded sum (a documented
    difference, DESIGN.md), so log-odds and the map are not compared; counters, indices, poses and weights are."""
    for wg, wo in zip(gpu.weights(), osl.weights()):
        assert np.array_equal(np.isnan(wg), np.isnan(wo))
    ref = _OddsFromDevice(osl, gpu) if saturated else _NanAsOne(osl)
    return compare_step(_NanAsOne(gpu), ref, check_map=not saturated)


def _sort_launches(cfg, scan, flags):
    """Launches of a step on a freshly uploaded scan minus those of a second step on the same scan: the beam sort
    runs once per scan, so this is 1 exactly when the step sorted the beams."""
    obs, odo = scan
    with GridMapSlam(cfg, GpuPlacement(seed=SEED, flags=flags)) as g:
        g.upload_scan(obs)
        before = g.launch_count
        g.step_async(odo)
        first = g.launch_count - before
        g.sync()
        before = g.launch_count
        g.step_async(odo)
        again = g.launch_count - before
        g.sync()
    return first - again


def _lockstep_stats(O, cfg, scans, flags):
    """common.lockstep, returning the handle's stats() after each step."""
    stats = []
    gpu = GridMapSlam(cfg, GpuPlacement(seed=SEED, flags=flags))
    osl = oracle_slam(O, cfg)
    try:
        for step, (obs, odo) in enumerate(scans):
            rc, _, _ = oracle_step(O, osl, obs, odo, step)
            assert rc == 0
            gpu.update(obs, odo)
            _compare(gpu, osl)
            stats.append(gpu.stats())
    finally:
        gpu.close()
        osl.close()
    return stats


def _lockstep_still(O, cfg, observations, poses, flags, saturated=False):
    """Lockstep with every particle held where it was placed: odometry (0, 0) and caller draws z = 0 move each particle
    by exactly 0 on both sides. Returns (stats(), oracle free counters of particle 0) per step."""
    n = cfg.n_particles
    odo = Odometry.new(0.0, 0.0, 0.1)
    z = np.zeros(2 * n)
    out = []
    gpu = GridMapSlam(cfg, GpuPlacement(seed=SEED, rng_mode=_lib.RNG_CALLER, flags=flags))
    osl = oracle_slam(O, cfg)
    try:
        gpu.set_poses(poses)
        osl.set_poses(poses)
        for step, obs in enumerate(observations):
            u = O.resample_uniform(SEED, step)
            ang = obs.angle.astype(f32).astype(np.float64)
            dist = obs.distance.astype(f32).astype(np.float64)
            assert osl.update(ang, dist, obs.valid.astype(np.uint8), f32(0.0), f32(0.0), f32(0.1), z, u) == 0
            gpu.update(obs, odo, z_draws=z, resample_u=u)
            _compare(gpu, osl, saturated)
            held = {tuple(p) for p in np.asarray(poses, f32).view(np.uint32)}
            assert {tuple(p) for p in gpu.poses().view(np.uint32)} <= held
            out.append((gpu.stats(), osl.counts(0)))
    finally:
        gpu.close()
        osl.close()
    return out


# ------------------------------------------------------------------------------------------------ 1. beam counts
@pytest.mark.parametrize("flags", ["default", "generic"])
@pytest.mark.parametrize("n_beams", [1, 32, 33, 2047, 2048, 2049, 4097])
def test_beam_count_thresholds(oracle, n_beams, flags):
    """Sorted for the ray kernel exactly when 32 < n <= 2048; packed and fused kernels up to 2047 beams, the 32-bit
    generic kernel above."""
    scans = make_scans(1.0, n_beams, 1.0, 3)
    assert all(len(obs) == n_beams for obs, _ in scans)
    if n_beams > 32:
        valid = np.concatenate([obs.valid for obs, _ in scans])
        assert valid.any() and not valid.all()
    lockstep(oracle, preset(), scans, flags=FLAGS[flags])
    assert _sort_launches(preset(), scans[0], FLAGS[flags]) == (1 if 32 < n_beams <= SORT_MAX_BEAMS else 0)


def test_beam_count_limit(oracle):
    """One step: every ray of the scan crosses the start cell, so 65,535 free hits fill its counter exactly; a second
    scan from nearby would saturate it (see test_zero_length_rays_saturate_the_generic_window for that)."""
    scans = make_scans(1.0, 65535, 1.0, 1)
    assert len(scans[0][0]) == 65535
    stats = _lockstep_stats(oracle, preset(), scans, 0)
    assert stats[0]["counter_saturated"] == 0
    assert _sort_launches(preset(), scans[0], 0) == 0


# ------------------------------------------------------------------------------------------------ 2. distances
def _band_edges(res):
    """Distances k res and (k +- 1) res, each with its f32 neighbours: where the classifier's thresholds switch."""
    out = []
    for k in (2, 10, 25):
        for m in (k - 1, k, k + 1):
            d = f32(m * res)
            out += [np.nextafter(d, f32(-1.0)), d, np.nextafter(d, f32(1e9))]
    return np.array(out, f32)


def _with_beams(obs, dist, valid, angle=None):
    n = len(dist)
    if angle is None:
        angle = np.arange(n, dtype=np.float64) * (2.0 * math.pi / n)
    return _obs(np.concatenate([obs.angle, angle]), np.concatenate([obs.distance, np.asarray(dist, np.float64)]),
                np.concatenate([obs.valid, np.asarray(valid, bool)]))


# Non-finite beams per scan. They walk to the grid border: from the start near the grid centre that is at least 100
# cells on the preset grid (window radius 50 + 6) and 256 on the 512^2 grid (radius 120 + 6), so every +-inf ray
# spends at least 44 (130) cells outside a window sized from the finite distances. The +-inf beams (two thirds) point
# in every direction, so each half of the disc receives at least 300 of them: on the 512^2 grid, whose tiled slots
# take the fused ray update, >= 300 x 130 = 39,000 window-bypassing hits per half-particle work item, far above the
# RAY_SPILL_CAP = 14,329 it can park (the 200^2 grid is not tiled: its packed kernel adds them to the grid directly).
N_NONFINITE = 900


def _degenerate(kind, scans, res):
    out = []
    for step, (obs, odo) in enumerate(scans):
        if kind == "nonfinite":
            vals = np.array([np.inf, -np.inf, np.nan], np.float64)[np.arange(N_NONFINITE) % 3]
            valid = (np.arange(N_NONFINITE) // 3 + step) % 2 == 0
            obs = _with_beams(obs, vals, valid)   # (beam 0 of these: +inf at angle 0)
            assert np.count_nonzero(np.isinf(vals)) // 2 * 130 > RAY_SPILL_CAP
        elif kind == "extremes":
            vals = np.array([0.0, -0.0, -0.3, -1e-3, -5.0, 1e-45, 1.4e-45, 1e30, -1e30, 3.0e38], np.float64)
            obs = _with_beams(obs, np.tile(vals, 4), np.arange(4 * vals.size) % 2 == step % 2)
        else:   # band edges
            vals = _band_edges(res).astype(np.float64)
            obs = _with_beams(obs, np.tile(vals, 4), np.arange(4 * vals.size) % 2 == 0)
        out.append((obs, odo))
    return out


def _geometry(name, n=8):
    if name == "preset_200":
        return preset(n), make_scans(1.0, 360, 1.0, 2)
    return at_scale_config(n), make_scans(10.0, 360, 6.0, 2)


@pytest.mark.parametrize("flags", ["default", "generic"])
@pytest.mark.parametrize("kind", ["nonfinite", "extremes", "band_edges"])
@pytest.mark.parametrize("geometry", ["preset_200", "at_scale_512"])
def test_degenerate_distances(oracle, geometry, kind, flags):
    cfg, base = _geometry(geometry)
    scans = _degenerate(kind, base, cfg.resolution)
    if kind == "nonfinite":
        assert len(scans[0][0]) <= RAY_PACKED_MAX_BEAMS   # the fused kernel's beam range
    stats = _lockstep_stats(oracle, cfg, scans, FLAGS[flags])
    if kind == "nonfinite" and geometry == "at_scale_512":   # (the 200^2 grid fits the largest window almost whole)
        assert stats and all(s["spilled_cells"] > 0 for s in stats), stats   # rays left the window


@pytest.mark.parametrize("flags", ["default", "generic"])
def test_infinite_beams_from_the_first_rows(oracle, flags):
    """Starts in column 0, rows 0 and 1, +inf beams toward +x+y: the reference's wrapping step count 3 + ax + ay gives
    1 cell from row 0 and 0 cells from row 1. Heading exactly 0, so +inf at angle 0 has ey = py + 0 x inf = NaN."""
    cfg = preset(8)
    res = cfg.resolution
    x0 = f32(cfg.position[0] + 0.5 * res)
    poses = np.array([[x0, f32(cfg.position[1] + (0.5 + (p % 2)) * res), 0.0] for p in range(8)], f32)
    ang = np.concatenate([[0.0], np.linspace(0.05, math.pi / 2 - 0.05, 60), [math.pi / 2]])
    dist = np.full(ang.size, np.inf)
    valid = np.arange(ang.size) % 2 == 0
    obs = _obs(ang, dist, valid)
    lockstep_out = _lockstep_still(oracle, cfg, [obs, obs], poses, FLAGS[flags])
    nf0, no0 = lockstep_out[-1][1]
    assert np.count_nonzero(nf0) + np.count_nonzero(no0) > 0


# ------------------------------------------------------------------------------------------------ 3. zero-length rays
ZL_CFG = GridMapSlamConfig(position=(-4.0, -4.0), width=8.0, height=8.0, resolution=0.25, n_particles=8)
ZL_POSE = (0.125, 0.125)   # (0.125 + 4) / 0.25 = 16.5 exactly: the centre of cell (16, 16)


def _zero_length_scan(n_beams, n_zero, n_zero_valid, rng_seed=3):
    """n_zero beams of distance 1e-9 (px + cos(a) 1e-9 rounds back to px: dx = dy = 0), the first n_zero_valid of
    them valid, and ordinary 1 m beams for the rest."""
    ang = np.arange(n_beams, dtype=np.float64) * (2.0 * math.pi / n_beams)
    dist = np.full(n_beams, 1.0)
    valid = np.arange(n_beams) % 2 == 0
    zl = np.random.default_rng(rng_seed).permutation(n_beams)[:n_zero]
    dist[zl] = 1e-9
    valid[zl] = False
    valid[zl[:n_zero_valid]] = True
    return _obs(ang, dist, valid)


def _start_cell(cfg, counts):
    gw = grid_cells(cfg.width, cfg.resolution)
    cx = int((ZL_POSE[0] - cfg.position[0]) / cfg.resolution)
    cy = int((ZL_POSE[1] - cfg.position[1]) / cfg.resolution)
    return int(counts[cy * gw + cx])


@pytest.mark.parametrize("flags", ["default", "generic"])
def test_zero_length_rays_overflow_the_packed_free_field(oracle, flags):
    """A zero-length ray emits its start cell three times. 1,747 of them (437 valid) and 300 ordinary beams put
    300 + 3 x 1,310 = 4,230 free hits on the start cell in one scan, beyond the packed window's 11-bit free field."""
    obs = _zero_length_scan(RAY_PACKED_MAX_BEAMS, 1747, 437)
    poses = np.array([[ZL_POSE[0], ZL_POSE[1], 0.0]] * ZL_CFG.n_particles, f32)
    out = _lockstep_still(oracle, ZL_CFG, [obs, obs], poses, FLAGS[flags])
    nf, no = out[0][1]
    assert _start_cell(ZL_CFG, nf) > RAY_PACKED_MAX_BEAMS
    assert _start_cell(ZL_CFG, no) == 3 * 437


def test_zero_length_rays_saturate_the_generic_window(oracle):
    """22,000 valid zero-length beams put 66,000 occupied hits on the start cell (any start offset) in one scan: the
    oracle saturates at 65,535, the 32-bit generic window's 16-bit occupied half must too."""
    n = 65535
    obs = _zero_length_scan(n, 22000, 22000)
    poses = np.array([[0.3, -0.2, 0.4]] * ZL_CFG.n_particles, f32)
    out = _lockstep_still(oracle, ZL_CFG, [obs], poses, _lib.FLAG_GENERIC_RAY_KERNEL, saturated=True)
    stats, (nf, no) = out[0]
    assert no.max() == 65535
    assert stats["counter_saturated"] > 0


# ------------------------------------------------------------------------------------------------ 4. device scans
def _device_scan(obs):
    a = torch.from_numpy(obs.angle.astype(f32)).cuda()
    d = torch.from_numpy(obs.distance.astype(f32)).cuda()
    v = torch.from_numpy(obs.valid.astype(np.uint8)).cuda()
    torch.cuda.synchronize()
    return a, d, v


def _true_max(obs):
    d = np.abs(obs.distance.astype(f32))
    return float(np.inf) if not np.all(np.isfinite(d)) else float(d.max(initial=0.0))


def _assert_same(a, b, particles):
    for wa, wb in zip(a.weights(), b.weights()):
        assert np.array_equal(wa.view(np.uint64), wb.view(np.uint64))
    assert np.array_equal(a.resample_indices(), b.resample_indices())
    assert np.array_equal(a.poses().view(np.uint32), b.poses().view(np.uint32))
    assert a.max_particle == b.max_particle
    assert a.estimated_pose() == b.estimated_pose()
    for p in particles:
        assert np.array_equal(a.cells(p), b.cells(p)), p


def _device_scans(case):
    if case.startswith("beams_"):
        return preset(), make_scans(1.0, int(case[6:]), 1.0, 2)
    geometry, kind = case.split(":")
    cfg, base = _geometry(geometry)
    return cfg, _degenerate(kind, base, cfg.resolution)


@pytest.mark.parametrize("max_dist", ["true", "inf", "nan", "zero"])
@pytest.mark.parametrize("case", ["beams_33", "beams_2047", "beams_4097", "preset_200:nonfinite", "preset_200:extremes",
                                  "at_scale_512:band_edges", "at_scale_512:nonfinite"])
def test_device_scan_equals_host_scan(case, max_dist):
    cfg, scans = _device_scans(case)
    with GridMapSlam(cfg, GpuPlacement(seed=SEED)) as dev, GridMapSlam(cfg, GpuPlacement(seed=SEED)) as host:
        for obs, odo in scans:
            md = {"true": _true_max(obs), "inf": float("inf"), "nan": float("nan"), "zero": 0.0}[max_dist]
            a, d, v = _device_scan(obs)
            dev.set_scan_device(a.data_ptr(), d.data_ptr(), v.data_ptr(), a.numel(), md)
            dev.step_async(odo)
            dev.sync()
            host.update(obs, odo)
            _assert_same(dev, host, (0, 3, cfg.n_particles - 1))
            del a, d, v


def test_device_scan_equals_host_scan_on_a_localizer():
    cfg = preset(129)
    prob = scene_map(reference_scene(1.0), cfg)
    scans = _localizer_scans(4096, "mixed", 2)
    with GridMapLocalizer(cfg, prob, MODELS["field"], GpuPlacement(seed=SEED)) as dev, \
            GridMapLocalizer(cfg, prob, MODELS["field"], GpuPlacement(seed=SEED)) as host:
        for obs, odo in scans:
            a, d, v = _device_scan(obs)
            dev.set_scan_device(a.data_ptr(), d.data_ptr(), v.data_ptr(), a.numel(), float("nan"))
            dev.step_async(odo)
            dev.sync()
            host.update(obs, odo)
            _assert_same(dev, host, ())
            del a, d, v


# ------------------------------------------------------------------------------------------------ 5. localiser windows
def _localizer_scans(n_beams, mask, steps, seed=11):
    """Simulator scans of n_beams beams with their valid masks replaced. 'mixed': the first window's valid count is
    not a multiple of 32, the second window (if any) has no valid beam, and some valid beams are non-finite (their
    endpoints fall off the grid). 'none': no valid beam at all."""
    rng = np.random.default_rng(seed)
    out = []
    for obs, odo in make_scans(1.0, n_beams, 1.0, steps):
        dist = obs.distance.copy()
        if mask == "none":
            valid = np.zeros(n_beams, bool)
        else:
            valid = rng.random(n_beams) < 0.6
            if n_beams > LOC_WIN:
                valid[LOC_WIN:2 * LOC_WIN] = False
            first = valid[:LOC_WIN]
            if np.count_nonzero(first) % 32 == 0:
                first[np.flatnonzero(first)[0]] = False
            idx = np.flatnonzero(valid)
            bad = idx[rng.permutation(idx.size)[:max(1, idx.size // 20)]]
            dist[bad] = np.array([np.inf, -np.inf, np.nan])[np.arange(bad.size) % 3]
        out.append((_obs(obs.angle, dist, valid), odo))
    return out


def _loc_lockstep(O, cfg, prob, model, scans):
    """As test_gpu_localize's driver: the oracle resamples on the device's raw weights once they have been checked
    against its own, so indices and poses must agree bit for bit."""
    n = cfg.n_particles
    g = grid_cells(cfg.width, cfg.resolution)
    ol = LO.OracleLocalizer(cfg.position, cfg.resolution, g, g, n, prob, model.kind, model.sigma, model.z_rand,
                            model.occupied_above)
    try:
        with GridMapLocalizer(cfg, prob, model, GpuPlacement(seed=SEED)) as loc:
            for step, (obs, odo) in enumerate(scans):
                z = O.motion_normals(SEED, step, 0, n)
                u = O.resample_uniform(SEED, step)
                loc.update(obs, odo)
                norm_g, raw_g = loc.weights()
                ol.set_weight_override(raw_g)
                ang = obs.angle.astype(f32).astype(np.float64)
                dist = obs.distance.astype(f32).astype(np.float64)
                assert ol.update(ang, dist, obs.valid.astype(np.uint8), f32(odo.distance_left),
                                 f32(odo.distance_right), f32(odo.wheel_distance), z, u) == 0
                assert _rel(raw_g, ol.own_raw_weights()) < WEIGHT_RTOL, step
                norm_o = ol.weights()[0]   # 0/0 = NaN when every raw weight underflows to 0, on both sides
                assert np.array_equal(np.isnan(norm_g), np.isnan(norm_o)), step
                assert _rel(np.nan_to_num(norm_g, nan=1.0), np.nan_to_num(norm_o, nan=1.0)) < WEIGHT_RTOL, step
                assert np.array_equal(loc.resample_indices().astype(np.int64), ol.indices().astype(np.int64)), step
                assert loc.max_particle == ol.max_particle
                assert np.array_equal(loc.poses().view(np.uint32), ol.poses().view(np.uint32)), step
                ep = loc.estimated_pose()
                assert np.array_equal(np.array([ep.x, ep.y, ep.theta], f32).view(np.uint32),
                                      ol.estimated_pose().view(np.uint32)), step
    finally:
        ol.close()


@pytest.mark.parametrize("mask", ["mixed", "none"])
@pytest.mark.parametrize("model", ["beam", "field"])
@pytest.mark.parametrize("n_beams", [1023, 1024, 1025, 2100, 4096, 65535])
def test_localizer_beam_windows(oracle, n_beams, model, mask):
    scans = _localizer_scans(n_beams, mask, 2)
    for obs, _ in scans:
        v = obs.valid
        if mask == "none":
            assert not v.any()
        else:
            assert np.count_nonzero(v[:LOC_WIN]) % 32 != 0
            assert np.any(v & ~np.isfinite(obs.distance))
            if n_beams > LOC_WIN:   # several windows, one of them without a valid beam
                assert not v[LOC_WIN:2 * LOC_WIN].any() and (n_beams <= 2 * LOC_WIN or v[2 * LOC_WIN:].any())
    prob = scene_map(reference_scene(1.0), preset())
    for n in (1, 31, 33, 129):   # partial warps and CTAs of k_loc_step
        _loc_lockstep(oracle, preset(n), prob, MODELS[model], scans)


@pytest.mark.parametrize("n_beams", [1025, 4096])
def test_beam_endpoint_localizer_equals_the_slam_step_across_windows(n_beams):
    """test_gpu_localize's bitwise cross-check with scans of several localiser windows: the SLAM step's k_likelihood
    folds the same terms in one pass, so raw weights must be bitwise equal."""
    n = 64
    cfg = preset(n)
    scans = make_scans(1.0, n_beams, 1.0, 4)
    with GridMapSlam(cfg, GpuPlacement(seed=SEED)) as a:
        for obs, odo in scans[:3]:
            a.update(obs, odo)
        cells = a.cells(a.max_particle)
        prob = a.estimated_likelihood()
        poses = a.poses()
    assert np.count_nonzero(cells) > 0
    rng = np.random.default_rng(7)
    z = rng.standard_normal(2 * n)
    u = 0.37
    obs, odo = scans[3]
    assert len(obs) == n_beams and obs.valid[:LOC_WIN].any() and obs.valid[LOC_WIN:].any()
    with GridMapSlam(cfg, GpuPlacement(seed=SEED, rng_mode=_lib.RNG_CALLER)) as b, \
            GridMapLocalizer(cfg, prob, SensorModel(), GpuPlacement(seed=SEED, rng_mode=_lib.RNG_CALLER)) as loc:
        for p in range(n):
            b.set_cells(p, cells)
        b.set_poses(poses)
        loc.set_poses(poses)
        b.update(obs, odo, z_draws=z, resample_u=u)
        loc.update(obs, odo, z_draws=z, resample_u=u)
        for wb, wl in zip(b.weights(), loc.weights()):
            assert np.array_equal(wb.view(np.uint64), wl.view(np.uint64))
        assert np.array_equal(b.resample_indices(), loc.resample_indices())
        assert np.array_equal(b.poses().view(np.uint32), loc.poses().view(np.uint32))
        assert b.estimated_pose() == loc.estimated_pose()


# ------------------------------------------------------------------------------------------------ 6. distance transform
DT_RES = 0.0625          # a power of two: w x DT_RES is exact, so the grid is exactly w cells wide
DT_MODEL = SensorModel.likelihood_field(sigma=0.1, z_rand=0.05, occupied_above=0.7)


def _field_terms(d2, model=DT_MODEL, res=DT_RES):
    """The likelihood-field term from exact squared distances in cells (NaN: no obstacle), in f64 numpy."""
    zr = float(f32(model.z_rand))
    zh = 1.0 - zr
    rr = float(f32(res)) * float(f32(res))
    ss = float(f32(model.sigma)) * float(f32(model.sigma))
    with np.errstate(invalid="ignore"):
        t = np.log(zh * np.exp(((-0.5 * d2) * rr) / ss) + zr)
    return np.where(np.isnan(d2), math.log(zr), t)


def _dt_map(w, kind):
    occ = float(f32(DT_MODEL.occupied_above))
    prob = np.full((w, w), 0.5)
    if kind == "corner_first":
        prob[0, 0] = 1.0
    elif kind == "corner_last":
        prob[w - 1, w - 1] = 1.0
    elif kind == "one_column":
        prob[:, w // 2] = 0.9
    elif kind == "one_row":
        prob[w // 3, :] = 0.9
    elif kind == "all":
        prob[:] = 1.0
    elif kind == "threshold":
        prob[:, :] = occ                                   # exactly at occupied_above: not an obstacle
        prob[(w - 1) // 2, w - 1] = np.nextafter(occ, 2.0)  # one step above it: an obstacle
    return prob


def _localizer_terms(w, prob):
    cfg = GridMapSlamConfig(position=(0.0, 0.0), width=w * DT_RES, height=w * DT_RES, resolution=DT_RES, n_particles=1)
    assert grid_cells(cfg.width, cfg.resolution) == w
    with GridMapLocalizer(cfg, prob.reshape(-1), DT_MODEL) as loc:
        return loc.sensor_terms().reshape(w, w)


@pytest.mark.parametrize("kind", ["none", "corner_first", "corner_last", "one_column", "one_row", "all", "threshold"])
@pytest.mark.parametrize("w", [1, 2, 255, 257])
def test_distance_transform_edges(w, kind):
    prob = _dt_map(w, kind)
    obstacle = prob > float(f32(DT_MODEL.occupied_above))
    if kind == "threshold":
        assert np.count_nonzero(obstacle) == 1
    if obstacle.any():
        d2 = np.rint(ndimage.distance_transform_edt(~obstacle) ** 2)
    else:
        d2 = np.full((w, w), np.nan)
    got = _localizer_terms(w, prob)
    ref = _field_terms(d2)
    if kind == "none":
        assert np.all(ref == math.log(float(f32(DT_MODEL.z_rand))))
    assert _rel(got, ref) < 1e-12


def test_distance_transform_wide_grid():
    """w = 12,289: the row pass keeps 4 x 12,289 = 49,156 bytes of column distances in shared memory, above the
    48 KB that needs no opt-in. 64 obstacles on a lattice; the reference is a brute force over them for 200 rows."""
    w = 12289
    assert 4 * w > 48 * 1024
    lat = np.linspace(37, w - 101, 8).astype(np.int64)
    oy, ox = (a.reshape(-1) for a in np.meshgrid(lat, lat + 13, indexing="ij"))
    prob = np.full((w, w), 0.5)
    prob[oy, ox] = 1.0
    got = _localizer_terms(w, prob)
    del prob
    rows = np.unique(np.concatenate([[0, w - 1], oy[:3], np.random.default_rng(5).choice(w, 197, replace=False)]))
    xs = np.arange(w, dtype=np.int64)
    worst = 0.0
    for y in rows:
        d2 = np.min((xs[:, None] - ox[None, :]) ** 2 + (int(y) - oy[None, :]) ** 2, axis=1).astype(np.float64)
        worst = max(worst, _rel(got[y], _field_terms(d2)))
    assert worst < 1e-12, worst
