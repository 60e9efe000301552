"""The chained step sequence (one GPU, device-resident scans, fused ray update: the ray update's last CTA joins the
planner and commits the step, profiling takes timestamps inside the kernels) against the serial one
(SLAMRS_FLAG_SERIAL_STEPS: events fork and join the planner, a separate kernel commits the step). Both run in one
process on the same scans, issued back to back with step_async and no host synchronisation in between; their state
must be equal bit for bit at every checkpoint. The oracle checks the chained sequence itself at a small size."""
from __future__ import annotations

import os
import re

import numpy as np
import pytest

from slamrs_b200 import GpuPlacement, GridMapSlam, GridMapSlamConfig, _lib
from slamrs_b200.workloads import WORKLOADS

from common import SEED, at_scale_config, at_scale_scans, compare_step, make_scans, oracle_slam, oracle_step

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_serial_steps_flag_in_header_and_binding():
    with open(os.path.join(ROOT, "include", "slamrs_gpu.h")) as f:
        m = re.search(r"SLAMRS_FLAG_SERIAL_STEPS\s*=\s*SLAMRS_FLAG_EAGER_COPY\s*<<\s*1\b", f.read())
    assert m and _lib.FLAG_EAGER_COPY << 1 == _lib.FLAG_SERIAL_STEPS == 32
    others = (_lib.FLAG_GENERIC_RAY_KERNEL, _lib.FLAG_UPDATE_ALL_PARTICLES, _lib.FLAG_FULL_GRID_COPY,
              _lib.FLAG_NCCL_EXCHANGE, _lib.FLAG_EAGER_COPY)
    assert all(_lib.FLAG_SERIAL_STEPS & f == 0 for f in others)


def _device_scans(scans):
    import torch
    out = []
    for obs, odo in scans:
        out.append((torch.from_numpy(obs.angle.astype(np.float32)).cuda(),
                    torch.from_numpy(obs.distance.astype(np.float32)).cuda(),
                    torch.from_numpy(obs.valid.astype(np.uint8)).cuda(),
                    float(np.abs(obs.distance.astype(np.float32)).max(initial=0.0)), odo))
    torch.cuda.synchronize()
    return out


def _issue(g, d_scans, lo, hi):
    for a, d, v, maxd, odo in d_scans[lo:hi]:
        g.set_scan_device(a.data_ptr(), d.data_ptr(), v.data_ptr(), a.numel(), maxd)
        g.step_async(odo)


def _state(g, particles):
    w, raw = g.weights()
    return {"w": w.view(np.uint64).copy(), "raw": raw.view(np.uint64).copy(), "idx": g.resample_indices(),
            "poses": g.poses().view(np.uint32).copy(), "max": g.max_particle,
            "pose": np.asarray([getattr(g.estimated_pose(), k) for k in ("x", "y", "theta")], np.float32).view(np.uint32),
            "map": g.estimated_likelihood().data.view(np.uint64).copy(),
            "cells": [g.cells(p).copy() for p in particles]}


def _assert_equal(a, b, where):
    for k in a:
        if k == "cells":
            for ca, cb in zip(a[k], b[k]):
                assert np.array_equal(ca, cb), where
        else:
            assert np.array_equal(np.asarray(a[k]), np.asarray(b[k])), (where, k)


def _chained_equals_serial(cfg, scans, checkpoints, slot_cells=0, tau=0.0, profiling=False):
    """Runs the scans through a chained and a serial filter (same process, same seed), back to back between
    checkpoints, and compares their state at each checkpoint; returns the launches per step of both."""
    d_scans = _device_scans(scans)
    pl = dict(seed=SEED, slot_cells=slot_cells, resample_threshold=tau)
    particles = (0, cfg.n_particles // 2, cfg.n_particles - 1)
    with GridMapSlam(cfg, GpuPlacement(**pl)) as chained, \
            GridMapSlam(cfg, GpuPlacement(flags=_lib.FLAG_SERIAL_STEPS, **pl)) as serial:
        launches = {}
        for g in (chained, serial):
            g.set_profiling(profiling)
        lo = 0
        for hi in checkpoints:
            for name, g in (("chained", chained), ("serial", serial)):
                before = g.launch_count
                _issue(g, d_scans, lo, hi)
                launches[name] = (g.launch_count - before) / (hi - lo)
            chained.sync()
            serial.sync()
            _assert_equal(_state(chained, particles), _state(serial, particles), hi)
            assert chained.stats() == serial.stats(), hi
            assert np.array_equal(chained.step_history(lo, hi - lo), serial.step_history(lo, hi - lo)), hi
            lo = hi
        if profiling:
            for g in (chained, serial):
                ph, n = g.phase_ms()
                assert n == checkpoints[-1] and all(v >= 0.0 for v in ph.values()), ph
                assert ph["ray_update"] > 0.0 and ph["motion_likelihood"] > 0.0, ph
    return launches


@pytest.mark.gpu
@pytest.mark.parametrize("n", [8192, 600, 4096], ids=["configs2", "items_just_above_ctas", "items_far_above_ctas"])
def test_chained_steps_equal_serial_steps(n):
    wl = WORKLOADS["c3"]
    cfg = wl.slam_config(n)
    sim = wl.simulator()
    scans = [sim.next_scan(wl.speed_left, wl.speed_right) for _ in range(210)]
    launches = _chained_equals_serial(cfg, scans, [1, 7, 64, 150, 210])
    assert launches["chained"] == launches["serial"] - 1   # no commit launch


@pytest.mark.gpu
def test_chained_steps_equal_serial_steps_windowed_slots():
    # (windowed slots take the unfused ray update, so both filters run the serial sequence: the flag changes nothing)
    wl = WORKLOADS["c5"]
    cfg = wl.slam_config(512)
    sim = wl.simulator()
    scans = [sim.next_scan(wl.speed_left, wl.speed_right) for _ in range(200)]
    _chained_equals_serial(cfg, scans, [5, 100, 200], slot_cells=wl.slot_cells)


@pytest.mark.gpu
def test_chained_steps_equal_serial_steps_adaptive_resampling():
    cfg = at_scale_config(2048)
    scans = at_scale_scans(200)
    _chained_equals_serial(cfg, scans, [3, 50, 200], tau=0.5)


@pytest.mark.gpu
def test_profiling_leaves_the_state_alone():
    cfg = at_scale_config(1024)
    scans = at_scale_scans(40)
    d_scans = _device_scans(scans)
    particles = (0, 511, 1023)
    with GridMapSlam(cfg, GpuPlacement(seed=SEED)) as on, GridMapSlam(cfg, GpuPlacement(seed=SEED)) as off:
        on.set_profiling(True)
        for g in (on, off):
            _issue(g, d_scans, 0, len(d_scans))
            g.sync()
        _assert_equal(_state(on, particles), _state(off, particles), "end")
        ph, n = on.phase_ms()
        assert n == len(d_scans) and ph["ray_update"] > 0.0
    _chained_equals_serial(cfg, scans[:20], [10, 20], profiling=True)


@pytest.mark.gpu
def test_chained_async_steps_lockstep_with_oracle(oracle):
    cfg = GridMapSlamConfig(position=(-4.0, -4.0), width=8.0, height=8.0, resolution=0.05, n_particles=64)
    scans = make_scans(3.0, 180, 3.0, 24)
    d_scans = _device_scans(scans)
    osl = oracle_slam(oracle, cfg)
    try:
        with GridMapSlam(cfg, GpuPlacement(seed=SEED)) as g:
            for lo, hi in ((0, 8), (8, 24)):
                _issue(g, d_scans, lo, hi)
                for step in range(lo, hi):
                    rc, _, _ = oracle_step(oracle, osl, *scans[step], step)
                    assert rc == 0
                g.sync()
                compare_step(g, osl)
    finally:
        osl.close()
