"""configs[4]'s shard in lockstep with the oracle: 720 beams, a 2048^2 grid at 5 cm in 512^2 windowed slots, a 6 m
lidar and uniform start poses over the 20 m room (workloads.uniform_poses on both sides), at 4,096 particles and, where
the host has the memory for the oracle's tiles, at the shard's full 32,768.

The room's centre, world (0, 0), is logical cell 1024 = 2 * 512, so the slots' torus seam runs through the middle of
the room on both axes and a large share of the particles have extents that wrap. One sparse oracle steps beside three
device handles -- deferred, eager and whole-grid copies -- and every handle is compared with the same oracle step
(common.lockstep_following_device_weights). Besides the fixed and most-cloned probes, each step compares particles
whose informed box straddles logical 1024 in x, in y and in both."""
import resource
import time

import numpy as np
import pytest

from slamrs_b200 import _lib
from slamrs_b200.workloads import WORKLOADS, uniform_poses

from common import cloned_probes, host_gib, lockstep_following_device_weights

pytestmark = pytest.mark.gpu

SEAM = 1024     # logical cell of world (0, 0): 2 * slot_cells
MODES = [0, _lib.FLAG_EAGER_COPY, _lib.FLAG_FULL_GRID_COPY]


def _straddle_probes(n):
    base = cloned_probes(n)
    seen = {"x": 0, "y": 0, "xy": 0, "fan_out": 0}

    def pick(step, idx, gpu):
        seen["fan_out"] = max(seen["fan_out"], int(np.bincount(idx).max()))
        out = set(base(step, idx))
        want = {"x", "y", "xy"}
        for p in range(n):
            if not want:
                break
            (x0, y0, x1, y1), _, _ = gpu.extents(p)
            sx, sy = x0 < SEAM < x1, y0 < SEAM < y1
            kind = "xy" if sx and sy else "x" if sx else "y" if sy else None
            if kind in want:
                want.discard(kind)
                seen[kind] += 1
                out.add(p)
        return sorted(out)
    return pick, seen


def _run(oracle, n):
    wl = WORKLOADS["c5"]
    cfg = wl.slam_config(n)
    sim = wl.simulator()
    scans = [sim.next_scan(wl.speed_left, wl.speed_right) for _ in range(4)]
    init = uniform_poses(wl, 0, n)

    def uniform_init(step, gpus, osl):
        if step == 0:
            for g in gpus:
                g.set_poses(init)
            osl.set_poses(init)

    probes, seen = _straddle_probes(n)
    t0 = time.monotonic()
    worst, surv, stats = lockstep_following_device_weights(oracle, cfg, scans, probes, check_map=True, flags=MODES,
                                                           slot_cells=wl.slot_cells, pre_step=uniform_init)
    wall = time.monotonic() - t0
    peak = resource.getrusage(resource.RUSAGE_SELF).ru_maxrss / 2 ** 20
    print(f"configs[4] shard lockstep at {n} particles: {wall:.1f} s for 4 scans, peak host RSS {peak:.1f} GiB, "
          f"worst weight error {worst:.2e}, survivors {surv}")
    # the geometry this file is for: boxes straddling the seam at logical 1024 on each axis and on both
    assert seen["x"] == seen["y"] == len(scans) and seen["xy"] > 0, seen
    # a copy job fans out to at most 16 destinations: some source has more clones than that
    assert seen["fan_out"] > 16, seen
    for step_stats in stats:
        for st in step_stats:
            assert st["window_overflow"] == 0, st
        eager = step_stats[MODES.index(_lib.FLAG_EAGER_COPY)]
        assert eager["grids_copied"] + eager["distinct_sources"] == n, eager
    return surv, stats


def test_configs4_shard_4096_particles(oracle):
    surv, stats = _run(oracle, 4096)
    assert 1 < surv[-1] < 4096


def test_configs4_shard_full_population(oracle):
    """The shard at its own population, 32,768 particles (262,144 on eight GPUs)."""
    if host_gib() < 64:
        pytest.skip("needs ~64 GiB of host memory for the oracle's tiles")
    surv, stats = _run(oracle, 32768)
    assert 1 < surv[-1] < 32768
