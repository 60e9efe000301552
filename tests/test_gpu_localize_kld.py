"""Adaptive population of the localiser (KLD-sampling, slamrs_gpu_set_kld): lockstep with the CPU oracle
(oracle/kld_oracle.c) for both sensor models, both RNG modes and recovery off and on; the generalised resampling pinned
to the fixed-size step at n_min = n_max = capacity; switching it on and off; hand-placed generations; device scans and
launch counts; the accessors' sizes and the argument checks; and global localisation at 2^20 particles."""
import ctypes as C
import math

import numpy as np
import pytest
import scipy.ndimage as ndi

from oracle import kld_oracle as KO
from slamrs_b200 import GpuPlacement, GridMapLocalizer, GridMapSlam, GridMapSlamConfig, Kld, Recovery, SensorModel, _lib, grid_cells
from slamrs_b200.simulator import Simulator, reference_scene, scene_map

from common import SEED, WEIGHT_RTOL, at_scale_config, make_scans

pytestmark = pytest.mark.gpu

PRESET = GridMapSlamConfig(position=(-2.0, -2.0), width=4.0, height=4.0, resolution=0.02, n_particles=256)
MODELS = {"beam": SensorModel(), "field": SensorModel.likelihood_field(sigma=0.1, z_rand=0.05)}
AGGRESSIVE = Recovery(alpha_slow=0.05, alpha_fast=0.5)
SCATTER_SEED = SEED + 1
KLD = {"preset": Kld(n_min=16, err=0.05, bin_xy=0.1, theta_bins=12),
       "at_scale": Kld(n_min=64, err=0.05, bin_xy=0.25, theta_bins=18)}


def room_map(segments, cfg, free_p=0.2):
    """scene_map with the 4-connected unknown region around the origin marked free (as the recovery tests do)."""
    g = grid_cells(cfg.width, cfg.resolution)
    prob = scene_map(segments, cfg)
    labels, _ = ndi.label((prob == 0.5).reshape(g, g))
    col = int(np.floor((0.0 - cfg.position[0]) / cfg.resolution))
    row = int(np.floor((0.0 - cfg.position[1]) / cfg.resolution))
    prob[(labels == labels[row, col]).reshape(-1)] = free_p
    return prob


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint64 if np.asarray(a).dtype == np.float64 else np.uint32)


def _tuple(kld, cfg):
    s = kld.to_struct(cfg.n_particles, cfg.resolution)
    return (s.n_min, s.n_max, s.err, s.z, s.bin_cells, s.theta_bins)


def _oracle_args(obs, odo):
    return (obs.angle.astype(np.float32).astype(np.float64), obs.distance.astype(np.float32).astype(np.float64),
            obs.valid.astype(np.uint8), np.float32(odo.distance_left), np.float32(odo.distance_right),
            np.float32(odo.wheel_distance))


def _lockstep(O, cfg, scene_scale, scan_range, model, rng_mode, kld, recovery, steps=10, scatter_at=5):
    """The localiser with KLD-sampling and the oracle side by side (the oracle resamples on the device's raw weights):
    N_t, k, M, the indices, the poses, the estimate and the recovery state bitwise equal at every step. Both start at
    Pose::default() (one bin: n_min), and the cloud is scattered over the room before step `scatter_at`, which makes
    the population grow again."""
    segments = reference_scene(scene_scale)
    prob = room_map(segments, cfg)
    scans = make_scans(scene_scale, 360, scan_range, steps)
    g = grid_cells(cfg.width, cfg.resolution)
    ol = KO.OracleKldLocalizer(cfg.position, cfg.resolution, g, g, cfg.n_particles, prob, model.kind, model.sigma,
                               model.z_rand, model.occupied_above)
    ol.set_kld(_tuple(kld, cfg))
    half = 0.9 * scene_scale
    trace = []
    with GridMapLocalizer(cfg, prob, model, GpuPlacement(seed=SEED, rng_mode=rng_mode)) as loc:
        loc.set_kld(kld)
        if recovery:
            loc.set_recovery(AGGRESSIVE)
            ol.set_recovery(AGGRESSIVE.alpha_slow, AGGRESSIVE.alpha_fast, SEED)
        for step, (obs, odo) in enumerate(scans):
            n = loc.population
            assert n == ol.population
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
            assert raw_g.size == n
            ol.set_weight_override(raw_g)
            assert ol.update(*_oracle_args(obs, odo), z, u) == 0
            own = ol.own_raw_weights()
            assert np.max(np.abs(raw_g - own) / np.maximum(np.abs(own), 1e-300)) < WEIGHT_RTOL, step
            st = loc.kld_state()
            assert (st["n_weighted"], st["k"], st["n_drawn"]) == ol.kld_state(), (step, st, ol.kld_state())
            assert loc.population == st["n_drawn"]
            assert np.array_equal(_bits(norm_g), _bits(ol.weights()[0])), step
            assert np.array_equal(loc.resample_indices().astype(np.int64), ol.indices().astype(np.int64)), step
            assert loc.max_particle == ol.max_particle
            assert np.array_equal(_bits(loc.poses()), _bits(ol.poses())), step
            ep = loc.estimated_pose()
            assert np.array_equal(_bits(np.array([ep.x, ep.y, ep.theta], np.float32)), _bits(ol.estimated_pose())), step
            if recovery:
                sg, so = loc.recovery_state(), ol.recovery_state()
                assert sg["injected"] == so["injected"], (step, sg, so)
                for key in ("w_slow", "w_fast", "p_inject"):
                    assert _bits(np.float64(sg[key])) == _bits(np.float64(so[key])), (step, key, sg, so)
            trace.append((st["n_weighted"], st["k"], st["n_drawn"]))
    ol.close()
    print("(N_t, k, M) per step:", trace)
    assert trace[0][2] == kld.n_min                       # one bin at Pose::default()
    n_t, _, m = trace[scatter_at]
    assert m > n_t or m == cfg.n_particles, trace            # the scattered cloud grows it again
    return trace


@pytest.mark.parametrize("recovery", [False, True])
@pytest.mark.parametrize("rng_mode", [_lib.RNG_SHARED_STREAM, _lib.RNG_CALLER])
@pytest.mark.parametrize("model", ["beam", "field"])
@pytest.mark.parametrize("geometry", ["preset_200", "at_scale_512"])
def test_kld_lockstep_with_oracle(oracle, geometry, model, rng_mode, recovery):
    if geometry == "preset_200":
        _lockstep(oracle, PRESET, 1.0, 1.0, MODELS[model], rng_mode, KLD["preset"], recovery)
    else:
        _lockstep(oracle, at_scale_config(4096), 10.0, 6.0, MODELS[model], rng_mode, KLD["at_scale"], recovery)


def _same_step(a, b):
    for wa, wb in zip(a.weights(), b.weights()):
        assert np.array_equal(_bits(wa), _bits(wb))
    assert np.array_equal(a.resample_indices(), b.resample_indices())
    assert np.array_equal(_bits(a.poses()), _bits(b.poses()))
    assert a.max_particle == b.max_particle
    assert a.estimated_pose() == b.estimated_pose()
    assert a.number_of_effective_particles() == b.number_of_effective_particles()


@pytest.mark.parametrize("recovery", [False, True])
def test_fixed_population_equals_kld_off(recovery):
    """n_min = n_max = capacity: every step is bitwise the fixed-size step, with one launch more."""
    cfg = at_scale_config(4096)
    prob = room_map(reference_scene(10.0), cfg)
    scans = make_scans(10.0, 360, 6.0, 6)
    with GridMapLocalizer(cfg, prob, MODELS["field"], GpuPlacement(seed=SEED)) as a, \
            GridMapLocalizer(cfg, prob, MODELS["field"], GpuPlacement(seed=SEED)) as b:
        b.set_kld(Kld(n_min=4096, n_max=4096))
        for h in (a, b):
            h.init_uniform((-4.0, -4.0, 4.0, 4.0))
            if recovery:
                h.set_recovery(AGGRESSIVE)
        for step, (obs, odo) in enumerate(scans):
            if step == 3:
                for h in (a, b):
                    h.init_uniform((-9.0, -9.0, 9.0, 9.0))
            la, lb = a.launch_count, b.launch_count
            a.update(obs, odo)
            b.update(obs, odo)
            assert b.launch_count - lb == a.launch_count - la + 1   # (update() also publishes the counters: one more)
            _same_step(a, b)
            st = b.kld_state()
            assert st["n_weighted"] == st["n_drawn"] == 4096 and st["k"] >= 1, st
            assert a.kld_state() == {"n_weighted": 0, "k": 0, "n_drawn": 0}
            if recovery:
                assert a.recovery_state() == b.recovery_state()


def test_switching_kld_on_and_off():
    cfg = at_scale_config(4096)
    prob = room_map(reference_scene(10.0), cfg)
    scans = make_scans(10.0, 360, 6.0, 8)
    with GridMapLocalizer(cfg, prob, MODELS["field"], GpuPlacement(seed=SEED)) as a, \
            GridMapLocalizer(cfg, prob, MODELS["field"], GpuPlacement(seed=SEED)) as b, \
            GridMapLocalizer(cfg, prob, MODELS["field"], GpuPlacement(seed=SEED)) as c:
        b.set_kld(KLD["at_scale"])
        b.set_kld(None)            # set and cleared before the first step: as if never set
        c.set_kld(KLD["at_scale"])
        for h in (a, b, c):
            h.init_uniform((-0.3, -0.3, 0.3, 0.3))
        for step, (obs, odo) in enumerate(scans):
            if step == 3:
                c.set_kld(None)
            n_c = c.population
            for h in (a, b, c):
                h.update(obs, odo)
            _same_step(a, b)
            assert a.population == b.population == 4096
            st = c.kld_state()
            if step < 3:
                assert st["n_weighted"] == n_c and st["n_drawn"] == c.population, st
                assert c.population < 4096
            else:   # cleared: the next step draws the capacity from N_t, and the handle stays there
                assert st == {"n_weighted": 0, "k": 0, "n_drawn": 0}
                assert c.weights()[0].size == n_c and c.population == 4096 and c.resample_indices().size == 4096
                assert int(c.resample_indices().max()) < n_c
            if step >= 4:
                assert n_c == 4096


def test_hand_placed_generations(oracle):
    cfg = at_scale_config(4096)
    g = grid_cells(cfg.width, cfg.resolution)
    prob = room_map(reference_scene(10.0), cfg)
    obs, odo = make_scans(10.0, 360, 6.0, 1)[0]
    kld = Kld(n_min=50, err=0.05, bin_xy=0.5, theta_bins=36)
    bc = kld.bin_cells(cfg.resolution)
    with GridMapLocalizer(cfg, prob, MODELS["field"], GpuPlacement(seed=SEED)) as loc:
        loc.set_kld(kld)
        # every pose in one bin: k = 1, n_min drawn
        loc.set_poses(np.tile(np.float32([0.11, -0.07, 0.2]), (4096, 1)))
        loc.update(obs, odo)
        assert loc.kld_state() == {"n_weighted": 4096, "k": 1, "n_drawn": 50} and loc.population == 50
        # poses on bin edges, just below them, off the grid and with edge headings: k as the oracle counts it
        res, x0 = np.float32(cfg.resolution), np.float32(cfg.position[0])
        cols = [0, bc - 1, bc, 2 * bc, g - 1, g, -1]
        xs = [x0 + np.float32(c) * res for c in cols] + [np.nextafter(x0 + np.float32(bc) * res, np.float32(-1e9))]
        thetas = [0.0, -0.0, math.pi, -math.pi, 2.0 * math.pi, float("inf"), float("nan"), -1e-30, 7.0]
        rng = np.random.default_rng(5)
        poses = np.array([[xs[i % len(xs)], xs[(i // 3) % len(xs)] - x0 + np.float32(cfg.position[1]),
                           thetas[i % len(thetas)]] for i in range(50)], np.float32)
        poses[rng.integers(0, 50, 5), 0] = np.float32("nan")
        loc.set_poses(poses)
        want_k = KO.kld_count(poses, cfg.position, cfg.resolution, g, g, bc, kld.theta_bins)
        loc.update(obs, odo)
        st = loc.kld_state()
        assert st["n_weighted"] == 50 and st["k"] == want_k > 5, (st, want_k)
        assert st["n_drawn"] == KO.kld_bound(want_k, 50, 4096, kld.err, kld.z) == loc.population
        # a population of 1 (n_min = 1, one bin) ...
        loc.set_kld(Kld(n_min=1, err=0.05))
        loc.set_poses(np.tile(np.float32([0.0, 0.0, 0.0]), (loc.population, 1)))
        loc.update(obs, odo)
        assert loc.population == 1
        # ... grows to n_max in one step, every draw from the one particle
        loc.set_kld(Kld(n_min=1000, n_max=1000))
        loc.update(obs, odo)
        assert loc.kld_state() == {"n_weighted": 1, "k": 1, "n_drawn": 1000}
        assert loc.population == 1000 and not loc.resample_indices().any()
        p = loc.poses()
        assert p.shape == (1000, 3) and np.all(_bits(p) == _bits(p[:1]))
        ep = loc.estimated_pose()
        assert np.array_equal(_bits(np.float32([ep.x, ep.y, ep.theta])), _bits(p[0]))


def test_device_scan_step_async_equals_update_and_launch_counts():
    cfg = at_scale_config(4096)
    segments = reference_scene(10.0)
    prob = room_map(segments, cfg)
    obs0, odo = make_scans(10.0, 360, 6.0, 1)[0]
    with GridMapLocalizer(cfg, prob, MODELS["field"], GpuPlacement(seed=SEED)) as a, \
            GridMapLocalizer(cfg, prob, MODELS["field"], GpuPlacement(seed=SEED)) as b:
        for h in (a, b):
            h.set_kld(KLD["at_scale"])
            h.init_uniform((-4.0, -4.0, 4.0, 4.0))
        for step in range(6):
            if step == 3:
                for h in (a, b):
                    h.set_recovery(AGGRESSIVE)
            pose = (0.1 * step, -0.2, 0.3 * step)
            a.sim_scan(segments, pose, 360, 6.0)
            before = a.launch_count
            a.step_async(odo)
            assert a.launch_count - before == (5 if step >= 3 else 4)
            a.sync()
            b.update(a.get_scan(), odo)
            _same_step(a, b)
            assert a.kld_state() == b.kld_state() and a.population == b.population
            if step >= 3:
                assert a.recovery_state() == b.recovery_state()
        a.set_profiling(True)
        for _ in range(4):
            a.step_async(odo)
        ms, steps = a.phase_ms()
        assert steps == 4 and ms["motion_likelihood"] > 0 and ms["resample"] > 0


def test_accessors_are_population_sized():
    cfg = at_scale_config(4096)
    prob = room_map(reference_scene(10.0), cfg)
    obs, odo = make_scans(10.0, 360, 6.0, 1)[0]
    with GridMapLocalizer(cfg, prob, MODELS["field"], GpuPlacement(seed=SEED, rng_mode=_lib.RNG_CALLER)) as loc:
        loc.set_kld(Kld(n_min=100, err=0.05))
        assert loc.population == 4096 and loc.poses().shape == (4096, 3)
        loc.set_poses(np.zeros((4096, 3), np.float32))
        z = np.random.default_rng(1).standard_normal(2 * 4096)
        with pytest.raises(ValueError):
            loc.update(obs, odo, z_draws=z[:100], resample_u=0.5)
        loc.update(obs, odo, z_draws=z, resample_u=0.5)
        assert loc.population == 100
        assert loc.poses().shape == (100, 3) and loc.resample_indices().shape == (100,)
        assert [w.shape for w in loc.weights()] == [(4096,), (4096,)]
        loc.init_uniform((-1.0, -1.0, 1.0, 1.0))
        p = loc.poses()
        assert p.shape == (100, 3) and np.all(np.abs(p[:, :2]) <= 1.0)
        with pytest.raises(ValueError):
            loc.step_async(odo, z_draws=z, resample_u=0.5)
        loc.upload_scan(obs)
        loc.step_async(odo, z_draws=z[:200], resample_u=0.5)
        loc.sync()
        assert [w.shape for w in loc.weights()] == [(100,), (100,)]
        assert 1.0 <= loc.number_of_effective_particles() <= 100.0


@pytest.mark.parametrize("what", ["slam", "threshold", "n_min_0", "n_min_above_n_max", "n_max_above_capacity", "err_0",
                                  "err_above_1", "err_nan", "z_negative", "z_inf", "bin_cells_0", "theta_bins_0",
                                  "theta_bins_3601", "bitmap", "struct_size"])
def test_set_kld_argument_checks(what):
    cfg = GridMapSlamConfig(position=(-2.0, -2.0), width=4.0, height=4.0, resolution=0.02, n_particles=256)
    if what == "bitmap":   # 512^2 cells x 3600 headings
        cfg = at_scale_config(256)
    prob = scene_map(reference_scene(1.0), cfg)
    k, msg = Kld(n_min=16), "KLD"
    if what == "slam":
        filt, msg = GridMapSlam(cfg), "SLAM handle"
    elif what == "threshold":
        filt, msg = GridMapLocalizer(cfg, prob, placement=GpuPlacement(resample_threshold=0.5)), "resample_threshold"
    elif what == "bitmap":
        filt, msg = GridMapLocalizer(cfg, prob), "2^28"
    else:
        filt = GridMapLocalizer(cfg, prob)
    s = k.to_struct(256, cfg.resolution)
    if what == "n_min_0": s.n_min = 0
    elif what == "n_min_above_n_max": s.n_min, s.n_max = 100, 99
    elif what == "n_max_above_capacity": s.n_max = 257
    elif what == "err_0": s.err = 0.0
    elif what == "err_above_1": s.err = 1.0 + 1e-12
    elif what == "err_nan": s.err = float("nan")
    elif what == "z_negative": s.z = -1e-9
    elif what == "z_inf": s.z = float("inf")
    elif what == "bin_cells_0": s.bin_cells = 0
    elif what == "theta_bins_0": s.theta_bins = 0
    elif what == "theta_bins_3601": s.theta_bins = 3601
    elif what == "bitmap": s.bin_cells, s.theta_bins = 1, 3600
    elif what == "struct_size": s.struct_size, msg = 32, "struct_size"
    with filt:
        rc = filt._L.slamrs_gpu_set_kld(filt._h, C.byref(s))
        assert rc == _lib.E_INVALID_ARG and msg.encode() in filt._L.slamrs_gpu_last_error(filt._h), \
            filt._L.slamrs_gpu_last_error(filt._h)
        if what == "slam":
            out = np.zeros(3, np.uint64)
            assert filt._L.slamrs_gpu_get_kld_state(filt._h, out.ctypes.data) == _lib.E_INVALID_ARG
            assert filt._L.slamrs_gpu_set_kld(filt._h, None) == _lib.E_INVALID_ARG
            n = C.c_uint64(0)
            assert filt._L.slamrs_gpu_get_population(filt._h, C.byref(n)) == _lib.OK and n.value == 256
        elif what != "threshold":   # the bounds themselves are valid, and NULL turns it off
            ok = Kld(n_min=1, n_max=256, err=1.0, z=0.0, bin_xy=0.1, theta_bins=3600 if what != "bitmap" else 1)
            filt.set_kld(ok)
            ok.bin_xy, ok.theta_bins = 1.0, 3600
            filt.set_kld(ok)
            filt.set_kld(None)
            assert filt.population == 256


# Global localisation at 2^20 particles: the scene and seed of test_global_localisation_from_a_uniform_start
# (tests/test_gpu_localize.py). The bounds come from one run on a B200 (DESIGN.md section 11.2): the population was
# n_min = 256 at every scan from the third on (330 at two of them), so twice n_min bounds it.
N_GLOBAL = 1 << 20
POP_BOUND_10_19 = 512


def _global(kld, scans=40):
    cfg = at_scale_config(N_GLOBAL)
    segments = reference_scene(5.0)
    sim = Simulator(segments, n_beams=360, scanner_range=6.0, wheel_base=0.1)
    trace = []
    with GridMapLocalizer(cfg, scene_map(segments, cfg), MODELS["field"], GpuPlacement(seed=SEED)) as loc:
        loc.set_kld(kld)
        loc.init_uniform((-4.5, -4.5, 4.5, 4.5))
        for _ in range(scans):
            obs, odo = sim.next_scan(0.08, 0.10)
            loc.update(obs, odo)
            ep = loc.estimated_pose()
            trace.append((round(math.hypot(ep.x - float(sim.pose[0]), ep.y - float(sim.pose[1])), 4),
                          round(abs(math.remainder(ep.theta - float(sim.pose[2]), 2.0 * math.pi)), 4),
                          loc.population, loc.kld_state()["k"]))
    return trace


def test_global_localisation_with_kld():
    """From a uniform start at 2^20 particles with Kld(): localised after 20 scans as the fixed-size filter is; the
    population over scans 10-19 stays below POP_BOUND_10_19; the mean position error over scans 20-39 is at most 1.5x
    the fixed-size run's, and the heading error stays below 0.05 rad. (The measured run: 0.050 m against 0.065 m; the
    heading error, 0.006 rad on average, is 2.4x the fixed-size run's 0.0024 rad.)"""
    adaptive = _global(Kld())
    fixed = _global(None)
    print("Kld() (err m, err rad, population, k) per scan:", adaptive)
    print("fixed 2^20 (err m, err rad):", [t[:2] for t in fixed])
    assert adaptive[19][0] < 0.2 and adaptive[19][1] < 0.15, adaptive[:20]
    assert max(t[2] for t in adaptive[10:20]) < POP_BOUND_10_19, adaptive[10:20]
    mean = lambda tr, j: sum(t[j] for t in tr[20:40]) / 20.0   # noqa: E731
    assert mean(adaptive, 0) <= 1.5 * mean(fixed, 0), (adaptive, fixed)
    assert max(t[1] for t in adaptive[20:40]) < 0.05, adaptive[20:40]
