"""Monte Carlo localisation against a loaded map (GridMapLocalizer / slamrs_gpu_create_localizer): lockstep with the
CPU oracle (oracle/loc_oracle.c) for both sensor models, an exact cross-check against the SLAM step's own likelihood,
global localisation from a uniform start, the localiser-only behaviour of the C ABI and one step at 2^20 particles."""
import math

import numpy as np
import pytest

from oracle import loc_oracle as LO
from slamrs_b200 import GpuPlacement, GridMapLocalizer, GridMapSlam, GridMapSlamConfig, SensorModel, _lib, grid_cells
from slamrs_b200.simulator import Simulator, reference_scene, scene_map

from common import SEED, WEIGHT_RTOL, at_scale_config, make_scans

pytestmark = pytest.mark.gpu

PRESET = GridMapSlamConfig(position=(-2.0, -2.0), width=4.0, height=4.0, resolution=0.02, n_particles=256)
MODELS = {"beam": SensorModel(), "field": SensorModel.likelihood_field(sigma=0.1, z_rand=0.05)}


def _rel(a, b):
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-300)))


def _oracle_localizer(cfg, prob, model):
    g = grid_cells(cfg.width, cfg.resolution)
    return LO.OracleLocalizer(cfg.position, cfg.resolution, g, g, cfg.n_particles, prob, model.kind, model.sigma,
                             model.z_rand, model.occupied_above)


def _lockstep(O, cfg, scene_scale, scan_range, model, rng_mode, steps=10, box=None, tau=0.0):
    """Runs the localiser and the oracle side by side; the oracle resamples on the device's raw weights after they
    have been checked against its own (slam_oracle.c so_set_weight_override), so indices must agree bit for bit."""
    prob = scene_map(reference_scene(scene_scale), cfg)
    scans = make_scans(scene_scale, 360, scan_range, steps)
    n = cfg.n_particles
    ol = _oracle_localizer(cfg, prob, model)
    ol.set_adaptive_resampling(tau)
    decisions = []
    with GridMapLocalizer(cfg, prob, model, GpuPlacement(seed=SEED, rng_mode=rng_mode, resample_threshold=tau)) as loc:
        assert _rel(loc.sensor_terms(), ol.terms()) < 1e-12
        if box is not None:
            loc.init_uniform(box)
            ol.set_poses(O.uniform_poses(SEED, 0, n, np.float32(box).astype(np.float64)))   # the device takes the box in f32
            assert np.array_equal(loc.poses().view(np.uint32), ol.poses().view(np.uint32))
        for step, (obs, odo) in enumerate(scans):
            z = O.motion_normals(SEED, step, 0, n)
            u = O.resample_uniform(SEED, step)
            if rng_mode == _lib.RNG_CALLER:
                loc.update(obs, odo, z_draws=z, resample_u=u)
            else:
                loc.update(obs, odo)
            norm_g, raw_g = loc.weights()
            ol.set_weight_override(raw_g)
            ang = obs.angle.astype(np.float32).astype(np.float64)
            dist = obs.distance.astype(np.float32).astype(np.float64)
            assert ol.update(ang, dist, obs.valid.astype(np.uint8), np.float32(odo.distance_left),
                             np.float32(odo.distance_right), np.float32(odo.wheel_distance), z, u) == 0
            assert _rel(raw_g, ol.own_raw_weights()) < WEIGHT_RTOL, step
            norm_o, _ = ol.weights()
            assert _rel(norm_g, norm_o) < WEIGHT_RTOL, step
            assert np.array_equal(loc.resample_indices().astype(np.int64), ol.indices().astype(np.int64)), step
            assert loc.max_particle == ol.max_particle
            assert np.array_equal(loc.poses().view(np.uint32), ol.poses().view(np.uint32)), step
            ep = loc.estimated_pose()
            assert np.array_equal(np.array([ep.x, ep.y, ep.theta], np.float32).view(np.uint32),
                                  ol.estimated_pose().view(np.uint32)), step
            assert abs(loc.number_of_effective_particles() - ol.number_of_effective_particles()) <= \
                WEIGHT_RTOL * ol.number_of_effective_particles()
            assert bool(loc.stats()["resampled"]) == ol.resampled()
            decisions.append(ol.resampled())
    ol.close()
    return decisions


@pytest.mark.parametrize("rng_mode", [_lib.RNG_SHARED_STREAM, _lib.RNG_CALLER])
@pytest.mark.parametrize("model", ["beam", "field"])
@pytest.mark.parametrize("geometry", ["preset_200", "at_scale_512"])
def test_lockstep_with_oracle(oracle, geometry, model, rng_mode):
    if geometry == "preset_200":
        _lockstep(oracle, PRESET, 1.0, 1.0, MODELS[model], rng_mode)
    else:
        _lockstep(oracle, at_scale_config(4096), 10.0, 6.0, MODELS[model], rng_mode)


@pytest.mark.parametrize("model", ["beam", "field"])
def test_lockstep_uniform_start(oracle, model):
    _lockstep(oracle, PRESET, 1.0, 1.0, MODELS[model], _lib.RNG_SHARED_STREAM, box=(-0.9, -0.9, 0.9, 0.9))


def test_lockstep_adaptive_resampling(oracle):
    decisions = []
    for model in ("beam", "field"):
        decisions += _lockstep(oracle, PRESET, 1.0, 1.0, MODELS[model], _lib.RNG_SHARED_STREAM, tau=0.5)
    assert any(decisions) and not all(decisions), decisions


def test_beam_endpoint_localizer_equals_the_slam_step_bit_for_bit():
    """A SLAM handle whose particles all hold grid C and a beam-endpoint localiser on C's probabilities score the same
    poses with the same draws: raw and normalised weights, indices, poses and the estimate are bitwise equal."""
    n = 64
    cfg = GridMapSlamConfig(position=(-2.0, -2.0), width=4.0, height=4.0, resolution=0.02, n_particles=n)
    scans = make_scans(1.0, 360, 1.0, 4)
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
        assert b.max_particle == loc.max_particle
        assert b.estimated_pose() == loc.estimated_pose()
        assert b.number_of_effective_particles() == loc.number_of_effective_particles()


def test_global_localisation_from_a_uniform_start():
    """Reference scene x5 (a 10 m room), 512^2 grid at 5 cm, 6 m lidar, likelihood field, 2^20 particles spread
    uniformly over the room: after 20 scans the estimate is within 0.2 m and 0.15 rad of the true pose."""
    cfg = at_scale_config(1 << 20)
    segments = reference_scene(5.0)
    sim = Simulator(segments, n_beams=360, scanner_range=6.0, wheel_base=0.1)
    errors = []
    with GridMapLocalizer(cfg, scene_map(segments, cfg), MODELS["field"], GpuPlacement(seed=SEED)) as loc:
        loc.init_uniform((-4.5, -4.5, 4.5, 4.5))
        for _ in range(20):
            obs, odo = sim.next_scan(0.08, 0.10)
            loc.update(obs, odo)
            ep = loc.estimated_pose()
            d_xy = math.hypot(ep.x - float(sim.pose[0]), ep.y - float(sim.pose[1]))
            d_th = abs(math.remainder(ep.theta - float(sim.pose[2]), 2.0 * math.pi))
            errors.append((round(d_xy, 4), round(d_th, 4)))
    print("global localisation error per step (m, rad):", errors)
    assert errors[-1][0] < 0.2 and errors[-1][1] < 0.15, errors


def test_grid_entry_points_fail_on_a_localizer():
    cfg = GridMapSlamConfig(position=(-2.0, -2.0), width=4.0, height=4.0, resolution=0.02, n_particles=32)
    with GridMapLocalizer(cfg, scene_map(reference_scene(1.0), cfg)) as loc:
        calls = [loc.estimated_likelihood, lambda: loc.estimated_likelihood_async(np.zeros(200 * 200)), loc.map_extent,
                 lambda: loc.estimated_likelihood_window((0, 0, 8, 8)), lambda: loc.cells(0),
                 lambda: loc.set_cells(0, np.zeros(200 * 200, np.uint32)), lambda: loc.log_odds(0), lambda: loc.extents(0),
                 loc.slots, lambda: loc.step_history(0, 1)]
        for call in calls:
            with pytest.raises(_lib.SlamrsGpuError) as e:
                call()
            assert e.value.code == _lib.E_INVALID_ARG and "a localizer has no particle grids" in str(e.value)
        assert loc.stats()["bytes_per_grid"] == 0
    with GridMapSlam(cfg) as slam:
        out = np.zeros(200 * 200)
        rc = slam._L.slamrs_gpu_get_sensor_terms(slam._h, out.ctypes.data)
        assert rc == _lib.E_INVALID_ARG and b"sensor-term table" in slam._L.slamrs_gpu_last_error(slam._h)


def test_three_launches_per_step_and_device_scan_equals_host_scan():
    cfg = at_scale_config(4096)
    segments = reference_scene(10.0)
    prob = scene_map(segments, cfg)
    obs0, odo = make_scans(10.0, 360, 6.0, 1)[0]
    with GridMapLocalizer(cfg, prob, MODELS["field"], GpuPlacement(seed=SEED)) as a, \
            GridMapLocalizer(cfg, prob, MODELS["field"], GpuPlacement(seed=SEED)) as b:
        a.init_uniform((-4.0, -4.0, 4.0, 4.0))
        b.init_uniform((-4.0, -4.0, 4.0, 4.0))
        for step in range(3):
            pose = (0.1 * step, -0.2, 0.3 * step)
            a.sim_scan(segments, pose, 360, 6.0)
            before = a.launch_count
            a.step_async(odo)
            assert a.launch_count - before == 3
            a.sync()
            b.update(a.get_scan(), odo)
            for wa, wb in zip(a.weights(), b.weights()):
                assert np.array_equal(wa.view(np.uint64), wb.view(np.uint64))
            assert np.array_equal(a.resample_indices(), b.resample_indices())
            assert np.array_equal(a.poses().view(np.uint32), b.poses().view(np.uint32))
            assert a.estimated_pose() == b.estimated_pose()
        a.set_profiling(True)
        for _ in range(4):
            a.step_async(odo)
        ms, steps = a.phase_ms()
        assert steps == 4 and ms["motion_likelihood"] > 0 and ms["resample"] > 0


def test_create_destroy_cycles_and_interleaving_with_slam(oracle):
    cfg = GridMapSlamConfig(position=(-2.0, -2.0), width=4.0, height=4.0, resolution=0.02, n_particles=64)
    prob = scene_map(reference_scene(1.0), cfg)
    scans = make_scans(1.0, 360, 1.0, 3)

    def slam_alone():
        with GridMapSlam(cfg, GpuPlacement(seed=SEED)) as s:
            for obs, odo in scans:
                s.update(obs, odo)
            return s.weights()[1], s.poses(), s.estimated_likelihood().data

    def loc_alone():
        with GridMapLocalizer(cfg, prob, MODELS["field"], GpuPlacement(seed=SEED)) as loc:
            for obs, odo in scans:
                loc.update(obs, odo)
            return loc.weights()[1], loc.poses()

    ref_slam, ref_loc = slam_alone(), loc_alone()
    for _ in range(3):
        assert all(np.array_equal(x, y) for x, y in zip(loc_alone(), ref_loc))
    with GridMapSlam(cfg, GpuPlacement(seed=SEED)) as s, \
            GridMapLocalizer(cfg, prob, MODELS["field"], GpuPlacement(seed=SEED)) as loc:
        for obs, odo in scans:
            s.update(obs, odo)
            loc.update(obs, odo)
        got_slam = (s.weights()[1], s.poses(), s.estimated_likelihood().data)
        got_loc = (loc.weights()[1], loc.poses())
    assert all(np.array_equal(x, y) for x, y in zip(got_slam, ref_slam))
    assert all(np.array_equal(x, y) for x, y in zip(got_loc, ref_loc))


def test_one_step_at_a_million_particles(oracle):
    n = 1 << 20
    cfg = at_scale_config(n)
    segments = reference_scene(10.0)
    prob = scene_map(segments, cfg)
    model = MODELS["field"]
    obs, odo = make_scans(10.0, 360, 6.0, 1)[0]
    box = (-4.5, -4.5, 4.5, 4.5)
    with GridMapLocalizer(cfg, prob, model, GpuPlacement(seed=SEED)) as loc:
        loc.init_uniform(box)
        start = loc.poses()
        loc.update(obs, odo)
        norm, raw = loc.weights()
        idx = loc.resample_indices()
        mp = loc.max_particle
    fold = oracle.resample_fold(raw, oracle.resample_uniform(SEED, 0))
    assert np.array_equal(idx.astype(np.int64), fold["idx"].astype(np.int64))
    assert mp == fold["max_particle"]
    assert _rel(norm, fold["norm"]) == 0.0
    sample = np.sort(np.random.default_rng(2024).choice(n, 2000, replace=False))
    ol = _oracle_localizer(GridMapSlamConfig(cfg.position, cfg.width, cfg.height, cfg.resolution, len(sample)),
                           prob, model)
    ol.set_poses(start[sample])
    z = np.concatenate([oracle.motion_normals(SEED, 0, int(p), 1) for p in sample])
    ang = obs.angle.astype(np.float32).astype(np.float64)
    dist = obs.distance.astype(np.float32).astype(np.float64)
    ol.update(ang, dist, obs.valid.astype(np.uint8), np.float32(odo.distance_left), np.float32(odo.distance_right),
              np.float32(odo.wheel_distance), z, 0.5)
    assert _rel(raw[sample], ol.own_raw_weights()) < WEIGHT_RTOL
    ol.close()
