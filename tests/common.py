"""Shared helpers of the parity tests: lockstep drivers for the GPU path and the CPU oracle."""
from __future__ import annotations

import os

import numpy as np

from slamrs_b200 import GpuPlacement, GridMapSlam, GridMapSlamConfig, Observation, Odometry
from slamrs_b200 import _lib
from slamrs_b200.simulator import Simulator, reference_scene
from slamrs_b200.slam import L_FREE, L_OCC

SEED = 0x5EED5A11
WEIGHT_RTOL = 1e-9   # stated tolerance of the contract is 1e-5 relative; we hold 1e-9
ODDS_RTOL = 1e-12


def gpu_present() -> bool:
    """Whether the CUDA driver reports a device (device node names differ between hosts and containers)."""
    import torch
    return torch.cuda.device_count() > 0


def make_scans(scene_scale, n_beams, scanner_range, steps, wheel_base=0.1, speed=(0.08, 0.10)):
    sim = Simulator(reference_scene(scene_scale), n_beams=n_beams, scanner_range=scanner_range, wheel_base=wheel_base)
    return [sim.next_scan(*speed) for _ in range(steps)]


def at_scale_config(n):
    """The bench's scene at half its grid side: 512^2 grids at 5 cm around a 20 m room, 6 m lidar."""
    return GridMapSlamConfig(position=(-12.8, -12.8), width=25.6, height=25.6, resolution=0.05, n_particles=n)


def at_scale_scans(steps):
    return make_scans(10.0, 360, 6.0, steps)


def host_gib() -> float:
    """MemAvailable of this host in GiB (0 when unknown): the oracle's tiles at full populations need tens of GiB."""
    try:
        with open("/proc/meminfo") as f:
            for line in f:
                if line.startswith("MemAvailable"):
                    return int(line.split()[1]) / 2 ** 20
    except OSError:
        pass
    return 0.0


def oracle_slam(O, cfg: GridMapSlamConfig, track_counts=True):
    return O.OracleSlam(cfg.position, cfg.width, cfg.height, cfg.resolution, cfg.n_particles, track_counts)


def oracle_step(O, osl, obs: Observation, odo: Odometry, step: int, seed=SEED):
    z = O.motion_normals(seed, step, 0, osl.n)
    u = O.resample_uniform(seed, step)
    # the reference casts angle/distance to f32 at use; feeding f32-representable f64 keeps both sides equal
    ang = obs.angle.astype(np.float32).astype(np.float64)
    dist = obs.distance.astype(np.float32).astype(np.float64)
    rc = osl.update(ang, dist, obs.valid.astype(np.uint8), np.float32(odo.distance_left), np.float32(odo.distance_right),
                    np.float32(odo.wheel_distance), z, u)
    return rc, z, u


def compare_step(gpu: GridMapSlam, osl, particles=None, check_map=True):
    """Asserts the parity contract after one lockstep update. Returns a dict of max errors."""
    n = osl.n
    w_ref, raw_ref = osl.weights()
    w_gpu, raw_gpu = gpu.weights()
    out = {}
    # resampled indices and ray cells: bit-exact
    idx_ref = osl.indices().astype(np.int64)
    idx_gpu = gpu.resample_indices().astype(np.int64)
    assert np.array_equal(idx_ref, idx_gpu), f"resample indices differ at {np.nonzero(idx_ref != idx_gpu)[0][:8]}"
    assert gpu.max_particle == osl.max_particle
    # poses: f32, bit-exact (same IEEE operations, same sin/cos)
    p_ref = osl.poses()
    p_gpu = gpu.poses()
    assert np.array_equal(p_ref.view(np.uint32), p_gpu.view(np.uint32)), "poses differ"
    # weights: f64 within tolerance (device exp/log differ from glibc by <= 1 ulp)
    den = np.maximum(np.abs(raw_ref), 1e-300)
    out["raw_weight_rel"] = float(np.max(np.abs(raw_gpu - raw_ref) / den))
    assert out["raw_weight_rel"] < WEIGHT_RTOL, out
    denn = np.maximum(np.abs(w_ref), 1e-300)
    out["norm_weight_rel"] = float(np.max(np.abs(w_gpu - w_ref) / denn))
    assert out["norm_weight_rel"] < WEIGHT_RTOL, out
    # grids: hit counters exact, reconstructed log-odds within tolerance
    particles = range(n) if particles is None else particles
    worst = 0.0
    for p in particles:
        nf_ref, no_ref = osl.counts(p)
        nf_gpu, no_gpu = gpu.counts(p)
        assert np.array_equal(nf_ref, nf_gpu), f"free counters differ for particle {p}"
        assert np.array_equal(no_ref, no_gpu), f"occupied counters differ for particle {p}"
        odds_ref = osl.odds(p)
        odds_gpu = gpu.log_odds(p)
        scale = np.maximum(np.abs(odds_ref), 1.0)
        worst = max(worst, float(np.max(np.abs(odds_gpu - odds_ref) / scale)))
    out["log_odds_rel"] = worst
    assert worst < ODDS_RTOL, out
    # published outputs
    ep_ref = osl.estimated_pose()
    ep = gpu.estimated_pose()
    assert np.array_equal(ep_ref.view(np.uint32), np.array([ep.x, ep.y, ep.theta], np.float32).view(np.uint32))
    if check_map:
        m_ref = osl.estimated_likelihood()
        m_gpu = gpu.estimated_likelihood().data
        out["map_abs"] = float(np.max(np.abs(m_ref - m_gpu)))
        assert out["map_abs"] < 1e-12, out
    return out


def lockstep(O, cfg: GridMapSlamConfig, scans, rng_mode=_lib.RNG_SHARED_STREAM, particles=None, seed=SEED, flags=0,
             pre_step=None, slot_cells=0):
    gpu = GridMapSlam(cfg, GpuPlacement(seed=seed, rng_mode=rng_mode, flags=flags, slot_cells=slot_cells))
    osl = oracle_slam(O, cfg)
    errs = []
    try:
        for step, (obs, odo) in enumerate(scans):
            if pre_step is not None:
                pre_step(step, gpu, osl)
            rc, z, u = oracle_step(O, osl, obs, odo, step, seed)
            assert rc == 0
            if rng_mode == _lib.RNG_CALLER:
                gpu.update(obs, odo, z_draws=z, resample_u=u)
            else:
                gpu.update(obs, odo)
            errs.append(compare_step(gpu, osl, particles))
    finally:
        gpu.close()
        osl.close()
    return errs


def install_cells(gpu: GridMapSlam, osl, particle: int, cells) -> None:
    """Installs one hand-built grid on both sides: packed hit counters (free | occupied << 16, index
    row * grid_h + column) into the device's slot and the same counters, with their log-odds, into the oracle
    (an oracle.scan_match_oracle.ScanMatchOracle; without a matcher set it is the plain oracle)."""
    c = np.ascontiguousarray(cells, np.uint32).reshape(-1)
    gpu.set_cells(particle, c)
    osl.set_counts(particle, (c & 0xFFFF).astype(np.uint16), (c >> 16).astype(np.uint16))


def lockstep_following_device_weights(O, cfg, scans, probes, check_map=True, flags=0, slot_cells=0, pre_step=None):
    """Lockstep of one sparse oracle with one device handle per entry of `flags` (an int or a sequence of flag
    sets), all on the same scans and seed. The device's exp/log differ from glibc's in the last bit, so raw weights
    agree to ~1e-12 relative, not bit for bit, and at large populations a resampling threshold lands that close to
    a prefix sum often enough to matter. Each step therefore (1) compares the oracle's own raw weights with the
    device's against WEIGHT_RTOL and (2) lets the oracle resample on the device's raw weights: on identical numbers
    the index vector, the argmax, every pose and every probed grid must then match bit for bit, on every handle.

    probes(step, idx, gpu) -> particles whose counters are compared (gpu: the first handle); pre_step(step, gpus,
    osl) runs before each step. Returns (worst relative weight error, distinct survivors per step, per step the
    list of every handle's stats())."""
    modes = list(flags) if isinstance(flags, (list, tuple)) else [flags]
    osl = O.OracleSlam(cfg.position, cfg.width, cfg.height, cfg.resolution, cfg.n_particles, True, sparse=True)
    osl.set_threads(os.cpu_count() or 1)
    worst_w = 0.0
    survivors, stats = [], []
    gpus = []
    try:
        for f in modes:
            gpus.append(GridMapSlam(cfg, GpuPlacement(seed=SEED, flags=f, slot_cells=slot_cells)))
        for step, (obs, odo) in enumerate(scans):
            if pre_step is not None:
                pre_step(step, gpus, osl)
            for g in gpus:
                g.update(obs, odo)
            w_gpu, raw_gpu = gpus[0].weights()
            for g in gpus[1:]:
                assert np.array_equal(g.weights()[1].view(np.int64), raw_gpu.view(np.int64)), (step, g.placement.flags)
            osl.set_weight_override(raw_gpu)
            rc, _, _ = oracle_step(O, osl, obs, odo, step)
            assert rc == 0
            own = osl.own_raw_weights()
            rel = np.max(np.abs(own - raw_gpu) / np.maximum(np.abs(own), 1e-300))
            worst_w = max(worst_w, float(rel))
            assert rel < WEIGHT_RTOL, (step, rel)
            w_ref, _ = osl.weights()
            idx_ref = osl.indices().astype(np.int64)
            survivors.append(len(np.unique(idx_ref)))
            p_ref = osl.poses().view(np.uint32)
            ep_ref = osl.estimated_pose().view(np.uint32)
            m_ref = osl.estimated_likelihood() if check_map else None
            picked = probes(step, idx_ref, gpus[0])
            counts_ref = {int(p): osl.counts(int(p)) for p in picked}
            step_stats = []
            for g in gpus:
                w_gpu = g.weights()[0]
                assert np.array_equal(w_ref.view(np.int64), w_gpu.view(np.int64)), "normalised weights differ on identical raw weights"
                idx_gpu = g.resample_indices().astype(np.int64)
                assert np.array_equal(idx_ref, idx_gpu), (step, g.placement.flags, np.nonzero(idx_ref != idx_gpu)[0][:8])
                assert g.max_particle == osl.max_particle
                assert np.array_equal(p_ref, g.poses().view(np.uint32)), (step, g.placement.flags)
                st = g.stats()
                assert st["resample_clamped"] == 0 and st["resample_exact_fallback"] == 0, st
                ep = g.estimated_pose()
                assert np.array_equal(ep_ref, np.array([ep.x, ep.y, ep.theta], np.float32).view(np.uint32))
                if check_map:
                    assert np.max(np.abs(m_ref - g.estimated_likelihood().data)) < 1e-12
                for p, (nf, no) in counts_ref.items():
                    gf, go = g.counts(p)
                    assert np.array_equal(nf, gf) and np.array_equal(no, go), (step, g.placement.flags, p)
                step_stats.append(st)
            stats.append(step_stats)
    finally:
        for g in gpus:
            g.close()
        osl.close()
    return worst_w, survivors, stats


def cloned_probes(n):
    """Probes for lockstep_following_device_weights: fixed particles, the most-cloned source's first and last
    copy, and a particle cloned exactly once."""
    def pick(step, idx, gpu=None):
        src, first, counts = np.unique(idx, return_index=True, return_counts=True)
        big = int(np.argmax(counts))
        out = {0, n // 2, n - 1, int(first[big]), int(first[big] + counts[big] - 1)}
        single = np.nonzero(counts == 1)[0]
        if single.size:
            out.add(int(first[single[0]]))
        return sorted(out)
    return pick
