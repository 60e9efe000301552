"""Lockstep against the oracle at BASELINE.json's real populations: configs[1] (1,024 x 360 x 512^2),
configs[2] (8,192 x 360 x 1024^2) and the population of configs[3] (65,536 particles) in one handle.

The oracle runs with tile storage and copy-on-write clones (same arithmetic as its dense layout, see
oracle/slam_oracle.c) because 8,192 dense f64 grids of 1024^2 cells would need 64 GiB. The device's
exp/log differ from glibc's in the last bit, so raw weights agree to ~1e-12 relative, not bit for bit;
at these populations a resampling threshold lands that close to a prefix sum often enough to matter.
Each step therefore (1) compares the oracle's own weights with the device's against the tolerance and
(2) lets the oracle resample on the device's raw weights -- on identical numbers the index vector, the
argmax, every pose and every probed grid must then match bit for bit (tests/test_gpu_resample_exact.py
covers the index kernels on adversarial weights)."""
import pytest

from slamrs_b200 import GridMapSlamConfig
from slamrs_b200.workloads import WORKLOADS

from common import cloned_probes, host_gib, lockstep_following_device_weights

pytestmark = pytest.mark.gpu


def test_lockstep_configs1_full_population(oracle):
    """configs[1]: 1,024 particles x 360 beams, 512^2 grid at 5 cm, 6 m range, 5 scans."""
    wl = WORKLOADS["c2"]
    cfg = wl.slam_config()
    sim = wl.simulator()
    scans = [sim.next_scan(wl.speed_left, wl.speed_right) for _ in range(5)]
    worst, surv, _ = lockstep_following_device_weights(oracle, cfg, scans, cloned_probes(cfg.n_particles))
    assert surv[-1] < cfg.n_particles


def test_lockstep_configs2_full_population(oracle):
    """configs[2]: 8,192 particles x 360 beams, 1024^2 grid, 4 scans (aliases, deferred copies and the
    survivors-only ray update all at the benchmark's own shape)."""
    if host_gib() < 24:
        pytest.skip("needs ~24 GiB of host memory for the oracle's tiles")
    wl = WORKLOADS["c3"]
    cfg = wl.slam_config()
    sim = wl.simulator()
    scans = [sim.next_scan(wl.speed_left, wl.speed_right) for _ in range(4)]
    worst, surv, _ = lockstep_following_device_weights(oracle, cfg, scans, cloned_probes(cfg.n_particles), check_map=True)
    assert 1 < surv[-1] < cfg.n_particles


def test_lockstep_configs3_population_in_one_handle(oracle):
    """65,536 particles (the population of configs[3]) in one handle on a small grid: the exact left folds,
    the index search and the planner at the 8-GPU population; 3 scans."""
    if host_gib() < 16:
        pytest.skip("needs ~16 GiB of host memory for the oracle's tiles")
    from slamrs_b200.simulator import Simulator, reference_scene
    n = 65536
    cfg = GridMapSlamConfig(position=(-6.4, -6.4), width=12.8, height=12.8, resolution=0.2, n_particles=n)
    sim = Simulator(reference_scene(5.0), n_beams=360, scanner_range=3.0, wheel_base=0.1)
    scans = [sim.next_scan(0.08, 0.10) for _ in range(3)]
    worst, surv, _ = lockstep_following_device_weights(oracle, cfg, scans, cloned_probes(n), check_map=True)
    assert 1 < surv[-1] < n
