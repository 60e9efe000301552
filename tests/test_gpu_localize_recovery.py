"""Recovery of the localiser from kidnapping and false convergence (augmented MCL, slamrs_gpu_set_recovery): lockstep
with the CPU oracle (oracle/recovery_oracle.c) for both sensor models and RNG modes, the unchanged step while recovery is
off, the injected poses at 2^20 particles against the stream's draws, the argument checks, and a kidnapped robot."""
import ctypes as C
import math

import numpy as np
import pytest
import scipy.ndimage as ndi

from oracle import recovery_oracle as RO
from slamrs_b200 import GpuPlacement, GridMapLocalizer, GridMapSlam, GridMapSlamConfig, Recovery, SensorModel, _lib, grid_cells
from slamrs_b200.simulator import Simulator, reference_scene, scene_map

from common import SEED, WEIGHT_RTOL, at_scale_config, make_scans

pytestmark = pytest.mark.gpu

PRESET = GridMapSlamConfig(position=(-2.0, -2.0), width=4.0, height=4.0, resolution=0.02, n_particles=256)
MODELS = {"beam": SensorModel(), "field": SensorModel.likelihood_field(sigma=0.1, z_rand=0.05)}
AGGRESSIVE = Recovery(alpha_slow=0.05, alpha_fast=0.5)
SCATTER_SEED = SEED + 1


def room_map(segments, cfg, free_p=0.2):
    """scene_map (walls 0.9, unknown 0.5) with the free space marked: the 4-connected unknown region around the origin
    (where the simulator starts) gets free_p. The walls close the room, so everything outside it stays unknown."""
    g = grid_cells(cfg.width, cfg.resolution)
    prob = scene_map(segments, cfg)
    labels, _ = ndi.label((prob == 0.5).reshape(g, g))
    col = int(np.floor((0.0 - cfg.position[0]) / cfg.resolution))
    row = int(np.floor((0.0 - cfg.position[1]) / cfg.resolution))
    prob[(labels == labels[row, col]).reshape(-1)] = free_p
    return prob


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint64 if np.asarray(a).dtype == np.float64 else np.uint32)


def _left_fold(values):
    s = 0.0
    for v in values.tolist():
        s += v
    return s


def _lockstep_recovery(O, cfg, scene_scale, scan_range, model, rng_mode, steps=10, scatter_at=5):
    """The localiser with recovery on and the oracle side by side; the oracle resamples on the device's raw weights
    (so_loc_set_weight_override), so its averages, its injections and every pose must agree bit for bit. The cloud is
    scattered over the room on both sides before step `scatter_at`, which makes the weights collapse."""
    segments = reference_scene(scene_scale)
    prob = room_map(segments, cfg)
    scans = make_scans(scene_scale, 360, scan_range, steps)
    n = cfg.n_particles
    g = grid_cells(cfg.width, cfg.resolution)
    ol = RO.OracleRecoveryLocalizer(cfg.position, cfg.resolution, g, g, n, prob, model.kind, model.sigma, model.z_rand,
                            model.occupied_above)
    ol.set_recovery(AGGRESSIVE.alpha_slow, AGGRESSIVE.alpha_fast, SEED)
    half = 0.9 * scene_scale
    trace = []
    with GridMapLocalizer(cfg, prob, model, GpuPlacement(seed=SEED, rng_mode=rng_mode)) as loc:
        loc.set_recovery(AGGRESSIVE)
        for step, (obs, odo) in enumerate(scans):
            if step == scatter_at:
                scatter = O.uniform_poses(SCATTER_SEED, 0, n, (-half, -half, half, half))
                loc.set_poses(scatter)
                ol.set_poses(scatter)
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
            own = ol.own_raw_weights()
            assert np.max(np.abs(raw_g - own) / np.maximum(np.abs(own), 1e-300)) < WEIGHT_RTOL, step
            st_g, st_o = loc.recovery_state(), ol.recovery_state()
            assert st_g["injected"] == st_o["injected"], (step, st_g, st_o)
            for key in ("w_slow", "w_fast", "p_inject"):
                assert _bits(np.float64(st_g[key])) == _bits(np.float64(st_o[key])), (step, key, st_g, st_o)
            assert np.array_equal(loc.resample_indices().astype(np.int64), ol.indices().astype(np.int64)), step
            assert loc.max_particle == ol.max_particle
            assert np.array_equal(_bits(loc.poses()), _bits(ol.poses())), step
            ep = loc.estimated_pose()
            assert np.array_equal(_bits(np.array([ep.x, ep.y, ep.theta], np.float32)), _bits(ol.estimated_pose())), step
            trace.append((st_g["p_inject"], st_g["injected"]))
    ol.close()
    print("(p_inject, injected) per step:", trace)
    assert any(k > 0 for _, k in trace) and any(k == 0 for _, k in trace), trace
    return trace


@pytest.mark.parametrize("rng_mode", [_lib.RNG_SHARED_STREAM, _lib.RNG_CALLER])
@pytest.mark.parametrize("model", ["beam", "field"])
@pytest.mark.parametrize("geometry", ["preset_200", "at_scale_512"])
def test_recovery_lockstep_with_oracle(oracle, geometry, model, rng_mode):
    if geometry == "preset_200":
        _lockstep_recovery(oracle, PRESET, 1.0, 1.0, MODELS[model], rng_mode)
    else:
        _lockstep_recovery(oracle, at_scale_config(4096), 10.0, 6.0, MODELS[model], rng_mode)


def test_recovery_off_means_the_step_is_unchanged():
    cfg = at_scale_config(4096)
    segments = reference_scene(10.0)
    prob = room_map(segments, cfg)
    scans = make_scans(10.0, 360, 6.0, 3)
    with GridMapLocalizer(cfg, prob, MODELS["field"], GpuPlacement(seed=SEED)) as a, \
            GridMapLocalizer(cfg, prob, MODELS["field"], GpuPlacement(seed=SEED)) as b:
        a.init_uniform((-4.0, -4.0, 4.0, 4.0))
        b.init_uniform((-4.0, -4.0, 4.0, 4.0))
        b.set_recovery(Recovery())
        b.set_recovery(None)
        for obs, odo in scans:
            a.update(obs, odo)
            b.update(obs, odo)
            for wa, wb in zip(a.weights(), b.weights()):
                assert np.array_equal(_bits(wa), _bits(wb))
            assert np.array_equal(a.resample_indices(), b.resample_indices())
            assert np.array_equal(_bits(a.poses()), _bits(b.poses()))
            assert a.estimated_pose() == b.estimated_pose()
            assert b.recovery_state() == {"w_slow": 0.0, "w_fast": 0.0, "p_inject": 0.0, "injected": 0}
        obs, odo = scans[0]
        a.upload_scan(obs)
        launches = []
        for rec in (None, Recovery(), None):
            a.set_recovery(rec)
            before = a.launch_count
            a.step_async(odo)
            launches.append(a.launch_count - before)
        a.sync()
        assert launches == [3, 4, 3]
        a.set_recovery(Recovery())
        a.set_profiling(True)
        for _ in range(4):
            a.step_async(odo)
        ms, steps = a.phase_ms()
        assert steps == 4 and ms["motion_likelihood"] > 0 and ms["resample"] > 0


def test_injected_poses_at_a_million_particles():
    """2^20 particles at the true pose, then scattered over the room: the weights collapse and p_inject is high. The
    averages equal the oracle's update on the device's raw sums; the injected count and every injected pose equal the
    stream's draws (ss_recovery_draw, oracle/recovery_oracle.c) bit for bit and lie in free cells; weights, indices, the estimate and every other
    pose equal those of a twin handle without recovery."""
    n = 1 << 20
    cfg = at_scale_config(n)
    segments = reference_scene(10.0)
    prob = room_map(segments, cfg)
    g = grid_cells(cfg.width, cfg.resolution)
    free = np.flatnonzero(prob < 0.5).astype(np.uint32)
    obs0, odo0 = make_scans(10.0, 360, 6.0, 1)[0]
    ws = wf = 0.0
    with GridMapLocalizer(cfg, prob, MODELS["field"], GpuPlacement(seed=SEED)) as loc, \
            GridMapLocalizer(cfg, prob, MODELS["field"], GpuPlacement(seed=SEED)) as twin:
        loc.set_recovery(AGGRESSIVE)
        for step in range(2):
            if step == 1:
                loc.init_uniform((-9.0, -9.0, 9.0, 9.0))
                twin.init_uniform((-9.0, -9.0, 9.0, 9.0))
            loc.update(obs0, odo0)
            twin.update(obs0, odo0)
            norm, raw = loc.weights()
            for a, b in zip((norm, raw), twin.weights()):
                assert np.array_equal(_bits(a), _bits(b))
            assert np.array_equal(loc.resample_indices(), twin.resample_indices())
            assert loc.estimated_pose() == twin.estimated_pose()
            ws, wf, p = RO.recovery_update(_left_fold(raw), n, AGGRESSIVE.alpha_slow, AGGRESSIVE.alpha_fast, ws, wf)
            st = loc.recovery_state()
            assert _bits(np.array([st["w_slow"], st["w_fast"], st["p_inject"]])).tolist() == \
                _bits(np.array([ws, wf, p])).tolist(), (step, st)
        assert st["p_inject"] > 0.3, st
        poses, resampled = loc.poses(), twin.poses()
    inject, draws = RO.recovery_draws(SEED, 1, 0, n, st["p_inject"], free, g, cfg.position, cfg.resolution)
    assert st["injected"] == int(inject.sum()) > 0.3 * n
    assert np.array_equal(_bits(poses[inject]), _bits(draws[inject]))
    # every injected pose lies in a free cell (a coordinate within an f32 rounding of a cell's upper edge may read as
    # the next cell: both candidates are tried)
    gx = (poses[inject, 0].astype(np.float64) - np.float32(cfg.position[0])) / np.float32(cfg.resolution)
    gy = (poses[inject, 1].astype(np.float64) - np.float32(cfg.position[1])) / np.float32(cfg.resolution)
    ok = np.zeros(gx.size, bool)
    for dx in (0.0, 1e-4):
        for dy in (0.0, 1e-4):
            ok |= prob[np.floor(gy - dy).astype(np.int64) * g + np.floor(gx - dx).astype(np.int64)] < 0.5
    assert ok.all()
    assert np.array_equal(_bits(poses[~inject]), _bits(resampled[~inject]))


@pytest.mark.parametrize("what", ["slam", "threshold", "no_free", "slow_0", "slow_eq_fast", "fast_above_1", "nan",
                                  "negative", "struct_size"])
def test_set_recovery_argument_checks(what):
    cfg = GridMapSlamConfig(position=(-2.0, -2.0), width=4.0, height=4.0, resolution=0.02, n_particles=64)
    segments = reference_scene(1.0)
    r = Recovery()
    if what == "slam":
        filt, msg = GridMapSlam(cfg), "SLAM handle"
    elif what == "threshold":
        filt, msg = GridMapLocalizer(cfg, room_map(segments, cfg), placement=GpuPlacement(resample_threshold=0.5)), \
            "resample_threshold"
    elif what == "no_free":
        filt, msg = GridMapLocalizer(cfg, scene_map(segments, cfg)), "free cells"
    else:
        filt, msg = GridMapLocalizer(cfg, room_map(segments, cfg)), "alpha"
        r = {"slow_0": Recovery(0.0, 0.1), "slow_eq_fast": Recovery(0.1, 0.1), "fast_above_1": Recovery(0.5, 1.0 + 1e-12),
             "nan": Recovery(float("nan"), 0.1), "negative": Recovery(-0.1, 0.1), "struct_size": Recovery()}[what]
    s = r.to_struct()
    if what == "struct_size":
        s.struct_size, msg = 16, "struct_size"
    with filt:
        rc = filt._L.slamrs_gpu_set_recovery(filt._h, C.byref(s))
        assert rc == _lib.E_INVALID_ARG and msg.encode() in filt._L.slamrs_gpu_last_error(filt._h), \
            filt._L.slamrs_gpu_last_error(filt._h)
        if what == "slam":
            out = np.zeros(3)
            assert filt._L.slamrs_gpu_get_recovery_state(filt._h, out.ctypes.data, None) == _lib.E_INVALID_ARG
        elif msg == "alpha":   # the bounds themselves are valid, and NULL turns recovery off
            filt.set_recovery(Recovery(1e-9, 1.0))
            filt.set_recovery(None)


N_KIDNAP = 1 << 20
KIDNAP_TO = (3.5, 3.0)   # metres: 1.5 m from the nearest wall of the 10 m room
KIDNAP_TURN = 2.0        # radians


def _kidnapped(recovery):
    """Reference scene x5 (10 m room), 512^2 at 5 cm, likelihood field, 6 m lidar: 20 scans from a uniform start, then
    the robot is carried to KIDNAP_TO and turned by KIDNAP_TURN without its odometry seeing it, then 40 more scans.
    Returns the per-step (error m, error rad, p_inject, injected)."""
    cfg = at_scale_config(N_KIDNAP)
    segments = reference_scene(5.0)
    sim = Simulator(segments, n_beams=360, scanner_range=6.0, wheel_base=0.1)
    trace = []
    with GridMapLocalizer(cfg, room_map(segments, cfg), MODELS["field"], GpuPlacement(seed=SEED)) as loc:
        loc.set_recovery(recovery)
        loc.init_uniform((-4.5, -4.5, 4.5, 4.5))
        for k in range(60):
            if k == 20:
                x, y, t = (float(v) for v in sim.pose)
                assert math.hypot(KIDNAP_TO[0] - x, KIDNAP_TO[1] - y) >= 3.0
                sim.pose = [np.float32(KIDNAP_TO[0]), np.float32(KIDNAP_TO[1]), np.float32(t + KIDNAP_TURN)]
            obs, odo = sim.next_scan(0.08, 0.10)
            loc.update(obs, odo)
            ep = loc.estimated_pose()
            st = loc.recovery_state()
            trace.append((round(math.hypot(ep.x - float(sim.pose[0]), ep.y - float(sim.pose[1])), 4),
                          round(abs(math.remainder(ep.theta - float(sim.pose[2]), 2.0 * math.pi)), 4),
                          float("%.4g" % st["p_inject"]), st["injected"]))
    return trace


def test_kidnapped_robot():
    """Localised after 20 scans with and without Recovery(), and bit for bit the same filter up to the kidnap (no
    injection while localised). Without recovery the filter stays lost. With Recovery() the kidnap is detected within
    the 40 scans -- late: w_slow has only reached about 1/40 of w_fast, which falls by a factor 0.9 per scan once the
    weights collapse and so needs some 35 scans to drop below it -- and the injected particles find the true pose again.
    The estimate does not settle in these scans: nothing resets the averages after an injection, so the injected
    particles lower the next mean weight and p_inject keeps rising (DESIGN.md section 11)."""
    with_rec = _kidnapped(Recovery())
    without = _kidnapped(None)
    print("with Recovery() (err m, err rad, p_inject, injected) per step:", with_rec)
    print("without recovery:", without)
    assert with_rec[:20] == without[:20] and with_rec[19][0] < 0.2 and with_rec[19][1] < 0.15, with_rec[:20]
    assert all(t[3] == 0 for t in with_rec[:20])
    assert all(t[0] > 1.0 for t in without[20:]) and all(t[3] == 0 for t in without), without
    first = next(i for i, t in enumerate(with_rec) if t[3] > 0)
    assert 20 < first < 59, with_rec
    assert any(t[0] < 0.2 and t[1] < 0.15 for t in with_rec[first:]), with_rec
