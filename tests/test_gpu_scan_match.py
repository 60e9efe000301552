"""Scan-matching pose refinement on the device (k_scan_match), in lockstep with the CPU oracle: poses, indices and
counters bit-exact, weights within 1e-9, and the four per-step statistics equal."""
from __future__ import annotations

import dataclasses
import os
import threading

import numpy as np
import pytest

from slamrs_b200 import (GpuPlacement, GridMapLocalizer, GridMapSlam, GridMapSlamConfig, Observation, Odometry,
                         ScanMatcher, _lib, nccl_unique_id)
from slamrs_b200.simulator import Simulator, reference_scene, scan, scene_map
from oracle.scan_match_oracle import ScanMatchOracle

from common import SEED, WEIGHT_RTOL, at_scale_config, at_scale_scans, compare_step, make_scans, oracle_step

pytestmark = pytest.mark.gpu

DEFAULT = ScanMatcher()


def oracle_slam(cfg, sparse=False):
    return ScanMatchOracle(cfg.position, cfg.width, cfg.height, cfg.resolution, cfg.n_particles, True, sparse=sparse)


def small_cfg(n=16):
    return GridMapSlamConfig(position=(-2.0, -2.0), width=4.0, height=4.0, resolution=0.02, n_particles=n)


def _stats_tuple(gpu):
    s = gpu.scan_match_stats()
    return (s["moved"], s["moves"], s["scored"], s["capped"])


def run(O, cfg, scans, matcher=DEFAULT, rng_mode=_lib.RNG_SHARED_STREAM, flags=0, slot_cells=0, tau=0.0,
        particles=None, pre_step=None, schedule=None, check_map=True, override=False, threads=1):
    """Lockstep with the matcher set on both sides (schedule(step) -> matcher or None overrides `matcher`).
    Returns the per-step stats and the per-step launch counts."""
    gpu = GridMapSlam(cfg, GpuPlacement(seed=SEED, rng_mode=rng_mode, flags=flags, slot_cells=slot_cells,
                                        resample_threshold=tau))
    osl = oracle_slam(cfg, sparse=override)
    osl.set_threads(threads)
    if tau:
        osl.set_adaptive_resampling(tau)
    stats, launches = [], []
    try:
        for step, (obs, odo) in enumerate(scans):
            if pre_step is not None:
                pre_step(step, gpu, osl)
            m = schedule(step) if schedule is not None else matcher
            gpu.set_scan_matcher(m)
            if m is None:
                osl.set_scan_match(levels=0)
            else:
                osl.set_scan_match(**dataclasses.asdict(m))
            l0 = gpu.launch_count
            if override:
                # large populations: both sides resample on the device's raw weights (see so_set_weight_override),
                # after those have been checked against the oracle's own
                gpu.update(obs, odo)
                raw_gpu = gpu.weights()[1]
                osl.set_weight_override(raw_gpu)
                assert oracle_step(O, osl, obs, odo, step)[0] == 0
                own = osl.own_raw_weights()
                assert np.max(np.abs(raw_gpu - own) / np.maximum(np.abs(own), 1e-300)) < WEIGHT_RTOL
            else:
                rc, z, u = oracle_step(O, osl, obs, odo, step)
                assert rc == 0
                if rng_mode == _lib.RNG_CALLER:
                    gpu.update(obs, odo, z_draws=z, resample_u=u)
                else:
                    gpu.update(obs, odo)
            launches.append(gpu.launch_count - l0)
            compare_step(gpu, osl, particles, check_map=check_map)
            st = _stats_tuple(gpu)
            assert st == osl.scan_match_stats(), (step, st, osl.scan_match_stats())
            stats.append(st)
    finally:
        gpu.close()
        osl.close()
    return stats, launches


def _total(stats, k):
    return sum(s[k] for s in stats)


# ------------------------------------------------------------------------------------------------ lockstep
@pytest.mark.parametrize("rng_mode", [_lib.RNG_SHARED_STREAM, _lib.RNG_CALLER], ids=["shared-stream", "caller"])
@pytest.mark.parametrize("radius", [0, 1, 2])
def test_lockstep_small_scene(oracle, radius, rng_mode):
    stats, _ = run(oracle, small_cfg(), make_scans(1.0, 360, 1.0, 8), dataclasses.replace(DEFAULT, radius=radius),
                   rng_mode=rng_mode)
    assert _total(stats, 1) > 0, "no particle moved"
    assert all(s[2] >= 16 * 7 for s in stats)


def test_lockstep_cap_and_border(oracle):
    """max_moves = 2 with coarse steps: particles stop at the cap. The grid ends 1 cell behind the room's walls, so
    radius-2 neighbourhoods of wall endpoints reach past the border."""
    cfg = GridMapSlamConfig(position=(-1.02, -1.02), width=2.04, height=2.04, resolution=0.02, n_particles=16)
    stats, _ = run(oracle, cfg, make_scans(1.0, 360, 1.5, 6),
                   ScanMatcher(radius=2, step_xy=0.02, step_theta=0.02, levels=2, max_moves=2))
    assert _total(stats, 3) > 0, "no particle reached max_moves"


def test_lockstep_at_scale(oracle):
    stats, _ = run(oracle, at_scale_config(1024), at_scale_scans(4), particles=[0, 511, 1023], check_map=False,
                   override=True, threads=os.cpu_count() or 1)
    assert _total(stats, 1) > 0


def test_lockstep_adaptive_resampling(oracle):
    stats, _ = run(oracle, small_cfg(32), make_scans(1.0, 360, 1.0, 8), tau=0.5)
    assert _total(stats, 1) > 0


@pytest.mark.parametrize("flags", [_lib.FLAG_FULL_GRID_COPY, _lib.FLAG_EAGER_COPY, _lib.FLAG_UPDATE_ALL_PARTICLES,
                                   _lib.FLAG_GENERIC_RAY_KERNEL],
                         ids=["full-grid-copy", "eager-copy", "update-all", "generic-ray"])
def test_lockstep_flags(oracle, flags):
    stats, _ = run(oracle, small_cfg(), make_scans(1.0, 360, 1.0, 6), flags=flags)
    assert _total(stats, 1) > 0


def test_lockstep_windowed_slots(oracle):
    """configs[4]'s shape at 20 particles (test_gpu_parity::test_c5_shape) with 512 x 512 windowed slots."""
    cfg = GridMapSlamConfig(position=(-51.2, -51.2), width=102.4, height=102.4, resolution=0.05, n_particles=20)
    scans = make_scans(10.0, 720, 6.0, 3)
    rng = np.random.default_rng(42)
    init = np.column_stack([rng.uniform(-9.0, 9.0, 20), rng.uniform(-9.0, 9.0, 20),
                            rng.uniform(-np.pi, np.pi, 20)]).astype(np.float32)

    def uniform_init(step, gpu, osl):
        if step == 0:
            gpu.set_poses(init); osl.set_poses(init)

    stats, _ = run(oracle, cfg, scans, particles=[0, 7, 19], pre_step=uniform_init, slot_cells=512, check_map=False)
    assert _total(stats, 1) > 0


def test_lockstep_many_beams_and_non_finite(oracle):
    scans = make_scans(1.0, 4096, 1.0, 4)
    obs, odo = scans[3]
    d = obs.distance.copy()
    v = np.nonzero(obs.valid)[0]
    d[v[::97]] = np.inf; d[v[13::97]] = np.nan; d[v[29::97]] = -np.inf
    scans[3] = (Observation(obs.id, angle=obs.angle, distance=d, valid=obs.valid), odo)
    assert int(np.sum(obs.valid)) > 2047
    stats, _ = run(oracle, small_cfg(8), scans)
    assert _total(stats, 1) > 0


# ------------------------------------------------------------------------------------------------ hand-built grids
def test_hand_built_grid_refines_to_the_true_pose(oracle):
    cfg = GridMapSlamConfig(position=(-1.5, -1.5), width=3.0, height=3.0, resolution=0.01, n_particles=8)
    segs = reference_scene(1.0)
    prob = scene_map(segs, cfg)
    n_occ = np.where(prob > 0.5, 3, 0).astype(np.uint32)
    n_free = np.where(prob > 0.5, 0, 1).astype(np.uint32)
    cells = n_free | (n_occ << 16)
    true = np.array([0.1, -0.2, 0.3], np.float32)
    start = true + np.array([0.04, -0.03, 0.03], np.float32)
    obs = scan(segs, true, 360, 2.0)
    odo = Odometry(0.0, 0.0, 0.1)   # zero draws below: the sample is the start pose
    m = ScanMatcher(radius=1, step_xy=0.08, step_theta=0.08, levels=4, max_moves=64)

    def place(step, gpu, osl):
        for p in range(cfg.n_particles):
            gpu.set_cells(p, cells)
            osl.set_counts(p, n_free.astype(np.uint16), n_occ.astype(np.uint16))
        gpu.set_poses(np.tile(start, (cfg.n_particles, 1))); osl.set_poses(np.tile(start, (cfg.n_particles, 1)))

    O = oracle
    gpu = GridMapSlam(cfg, GpuPlacement(seed=SEED, rng_mode=_lib.RNG_CALLER))
    osl = oracle_slam(cfg)
    try:
        place(0, gpu, osl)
        gpu.set_scan_matcher(m); osl.set_scan_match(**dataclasses.asdict(m))
        z = np.zeros(2 * cfg.n_particles)
        ang = obs.angle.astype(np.float32).astype(np.float64); dist = obs.distance.astype(np.float32).astype(np.float64)
        assert osl.update(ang, dist, obs.valid.astype(np.uint8), 0.0, 0.0, 0.1, z, 0.5) == 0
        gpu.update(obs, odo, z_draws=z, resample_u=0.5)
        compare_step(gpu, osl)
        assert _stats_tuple(gpu) == osl.scan_match_stats()
        assert _stats_tuple(gpu)[0] == cfg.n_particles
        poses = gpu.poses()
        assert np.all(np.abs(poses[:, :2] - true[:2]) <= 0.01 + 1e-6), poses
        assert np.all(np.abs(poses[:, 2] - true[2]) <= 0.01 + 1e-6), poses
    finally:
        gpu.close(); osl.close()


# ------------------------------------------------------------------------------------------------ switching
def test_switching_on_and_off(oracle):
    scans = make_scans(1.0, 360, 1.0, 7)
    on_steps = {2, 3, 4}
    stats, launches = run(oracle, small_cfg(), scans, schedule=lambda s: DEFAULT if s in on_steps else None)
    with GridMapSlam(small_cfg(), GpuPlacement(seed=SEED)) as ref:
        base = []
        for obs, odo in scans:
            l0 = ref.launch_count
            ref.update(obs, odo)
            base.append(ref.launch_count - l0)
    for step in range(len(scans)):
        assert launches[step] == base[step] + (1 if step in on_steps else 0), (step, launches, base)
        if step not in on_steps:
            assert stats[step] == (0, 0, 0, 0)
    assert sum(stats[s][1] for s in on_steps) > 0


def test_argument_checks_and_localizer():
    with GridMapSlam(small_cfg(4), GpuPlacement(seed=SEED)) as g:
        for bad in [dict(radius=3), dict(step_xy=0.0), dict(step_xy=float("inf")), dict(step_theta=float("nan")),
                    dict(levels=0), dict(levels=9), dict(max_moves=0), dict(max_moves=1025)]:
            with pytest.raises(_lib.SlamrsGpuError) as e:
                g.set_scan_matcher(dataclasses.replace(DEFAULT, **bad))
            assert e.value.code == _lib.E_INVALID_ARG
        bad = DEFAULT.to_struct(); bad.struct_size = 20
        import ctypes as C
        assert g._L.slamrs_gpu_set_scan_match(g._h, C.byref(bad)) == _lib.E_INVALID_ARG
        g.set_scan_matcher(None)
        assert g.scan_match_stats() == dict(moved=0, moves=0, scored=0, capped=0)
    cfg = small_cfg(4)
    loc = GridMapLocalizer(cfg, scene_map(reference_scene(1.0), cfg))
    try:
        with pytest.raises(_lib.SlamrsGpuError) as e:
            loc.set_scan_matcher(DEFAULT)
        assert e.value.code == _lib.E_INVALID_ARG
    finally:
        loc.close()


# ------------------------------------------------------------------------------------------------ quality
QUALITY_FROM = 20   # scans over which the error is averaged (the map has content by then)


def quality_run(matcher, n=64, steps=40):
    """configs[1]'s scene: scale 5, 6 m lidar, 512^2 grid at 5 cm. Returns per-scan (position, heading) errors of
    estimated_pose() against the simulator's pose."""
    cfg = GridMapSlamConfig(position=(-12.8, -12.8), width=25.6, height=25.6, resolution=0.05, n_particles=n)
    sim = Simulator(reference_scene(5.0), n_beams=360, scanner_range=6.0, wheel_base=0.1)
    errs = []
    with GridMapSlam(cfg, GpuPlacement(seed=SEED)) as g:
        g.set_scan_matcher(matcher)
        for _ in range(steps):
            obs, odo = sim.next_scan(0.08, 0.10)
            g.update(obs, odo)
            ep = g.estimated_pose()
            true = [float(v) for v in sim.pose]
            dth = (ep.theta - true[2] + np.pi) % (2 * np.pi) - np.pi
            errs.append((float(np.hypot(ep.x - true[0], ep.y - true[1])), abs(float(dth))))
    return np.array(errs)


def test_quality_matcher_lowers_the_pose_error():
    off = quality_run(None)[QUALITY_FROM:].mean(axis=0)
    on = quality_run(DEFAULT)[QUALITY_FROM:].mean(axis=0)
    print(f"mean error over scans {QUALITY_FROM}-39, matcher off: {off[0]:.4f} m {off[1]:.4f} rad; "
          f"on: {on[0]:.4f} m {on[1]:.4f} rad")
    # measured on a B200 (the run is deterministic): position 0.0511 m -> 0.0262 m, heading 0.0180 -> 0.0217 rad. The
    # matcher halves the position error; at these defaults it does not lower the heading error (see DESIGN.md).
    assert on[0] < 0.7 * off[0], (on, off)
    assert on[1] < 1.5 * off[1], (on, off)


# ------------------------------------------------------------------------------------------------ two GPUs
def test_two_gpus_lockstep(oracle):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    world, n = 2, 32
    cfg = small_cfg(n)
    scans = make_scans(1.0, 360, 1.0, 6)
    nid = nccl_unique_id()
    out, errs = [None] * world, []

    def worker(rank):
        g = None
        try:
            g = GridMapSlam(cfg, GpuPlacement(device=rank, rank=rank, world_size=world, nccl_id=nid, seed=SEED))
            g.set_scan_matcher(DEFAULT)
            rec = []
            for obs, odo in scans:
                g.update(obs, odo)
                rec.append(dict(poses=g.poses().copy(), idx=g.resample_indices().copy(), stats=_stats_tuple(g)))
            out[rank] = rec
        except Exception as e:  # noqa: BLE001
            errs.append((rank, repr(e)))
        finally:
            if g is not None:
                g.close()

    ts = [threading.Thread(target=worker, args=(r,)) for r in range(world)]
    [t.start() for t in ts]
    [t.join(timeout=120) for t in ts]
    assert not errs, errs
    assert all(o is not None for o in out), "a rank hung"
    osl = oracle_slam(cfg)
    osl.set_scan_match(**dataclasses.asdict(DEFAULT))
    moved = 0
    for step, (obs, odo) in enumerate(scans):
        assert oracle_step(oracle, osl, obs, odo, step)[0] == 0
        poses = osl.poses()
        for r in range(world):
            rec = out[r][step]
            assert np.array_equal(rec["idx"], osl.indices().astype(np.uint32))
            lo = r * (n // world)
            assert np.array_equal(rec["poses"].view(np.uint32), poses[lo:lo + n // world].view(np.uint32))
        summed = tuple(sum(out[r][step]["stats"][k] for r in range(world)) for k in range(4))
        assert summed == osl.scan_match_stats()
        moved += summed[0]
    assert moved > 0
    osl.close()
