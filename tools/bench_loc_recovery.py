"""Cost of the localiser's recovery (augmented MCL, slamrs_gpu_set_recovery) on one B200: the device time of one
step_async at configs[2]'s scene (20 m room, 1024^2 at 5 cm with the room's free space marked, 6 m lidar, 360 beams,
likelihood field) for 8,192, 262,144 and 1,048,576 particles, three ways:

    off      no recovery (three launches per step)
    p = 0    recovery on, alpha_slow = 1e-9 and alpha_fast = 1: a first step on a cloud scattered over the room seeds
             w_slow with a tiny mean weight, then the particles are put at the true pose; w_fast follows the (much
             larger) mean weight and w_slow hardly moves, so p stays 0 (k_loc_recover returns before any draw). The
             off leg runs the same sequence, so both time the same cloud
    p high   recovery on (0.05 / 0.5), particles first at the true pose, then scattered over the room: the mean weight
             collapses and stays low, so p stays near 1 and almost every particle takes a Philox draw and a new pose

The robot stands still (zero odometry, the same scan every step). The time of k_loc_step depends on where the
particles are (the term-table gathers), so the p high leg, whose cloud is a new uniform one every step, is compared
by the resample phase (k_weights + k_resample_indices + k_loc_recover, CUDA events) rather than by the whole step.

Each leg reports the p_inject and injected counts of its timed steps. Card and power limit are read in the same run.
Writes profiles/loc_recovery_1gpu.json (or --out). Needs a GPU: there is no fallback.

    python tools/bench_loc_recovery.py [--steps 50] [--warmup 5] [--out profiles/loc_recovery_1gpu.json]
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_localize import card  # noqa: E402
from slamrs_b200 import GpuPlacement, GridMapLocalizer, Odometry, Recovery, SensorModel  # noqa: E402
from slamrs_b200.workloads import WORKLOADS  # noqa: E402
from test_gpu_localize_recovery import room_map  # noqa: E402

SEED = 0x5EED5A11
MODEL = SensorModel.likelihood_field(sigma=0.1, z_rand=0.05)
LEGS = {"off": None, "p0": Recovery(alpha_slow=1e-9, alpha_fast=1.0), "p_high": Recovery(alpha_slow=0.05, alpha_fast=0.5)}


def timed(loc, odo, steps, warmup):
    """Per-step device time (CUDA events around each step_async on the handle's stream) and the recovery state of
    every timed step."""
    import torch
    stream = torch.cuda.ExternalStream(loc.stream_ptr)
    for _ in range(warmup):
        loc.step_async(odo)
    loc.sync()
    times, p, injected = [], [], []
    for _ in range(steps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        loc.step_async(odo)
        b.record(stream)
        b.synchronize()
        times.append(a.elapsed_time(b))
        st = loc.recovery_state()
        p.append(st["p_inject"])
        injected.append(st["injected"])
    return times, p, injected


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "loc_recovery_1gpu.json"))
    args = ap.parse_args()
    import torch
    if torch.cuda.device_count() == 0:
        raise SystemExit("bench_loc_recovery: no GPU visible (the localiser has no CPU path)")
    wl = WORKLOADS["c3"]
    sim = wl.simulator()
    obs, _ = sim.next_scan(wl.speed_left, wl.speed_right)
    odo = Odometry(0.0, 0.0, wl.wheel_base)
    truth = np.array([[float(v) for v in sim.pose]], np.float32)
    half = 0.9 * wl.scene_scale
    result = {"card": card(), "steps": args.steps, "warmup": args.warmup, "workload": "c3 scene, likelihood field",
              "rows": []}
    for n in (8192, 262144, 1 << 20):
        cfg = wl.slam_config(n)
        prob = room_map(sim.segments, cfg)
        for leg, rec in LEGS.items():
            with GridMapLocalizer(cfg, prob, MODEL, GpuPlacement(seed=SEED)) as loc:
                loc.set_recovery(rec)
                loc.upload_scan(obs)
                at_truth = np.repeat(truth, n, axis=0)
                if leg == "p_high":
                    loc.set_poses(at_truth)
                    loc.step_async(odo)
                    loc.init_uniform((-half, -half, half, half))
                else:
                    loc.init_uniform((-half, -half, half, half))
                    loc.step_async(odo)
                    loc.set_poses(at_truth)
                before = loc.launch_count
                loc.step_async(odo)
                launches = loc.launch_count - before
                times, p, injected = timed(loc, odo, args.steps, args.warmup)
                loc.set_profiling(True)
                for _ in range(args.steps):
                    loc.step_async(odo)
                ms, k = loc.phase_ms()
                loc.set_profiling(False)
            row = {"n_particles": n, "leg": leg, "launches_per_step": launches, "step_ms_median": float(np.median(times)),
                   "step_ms_min": float(np.min(times)), "step_ms_max": float(np.max(times)),
                   "k_loc_step_ms": ms["motion_likelihood"] / k, "resample_phase_ms": ms["resample"] / k,
                   "p_inject_min": float(np.min(p)), "p_inject_max": float(np.max(p)),
                   "injected_mean": float(np.mean(injected))}
            result["rows"].append(row)
            print(row, flush=True)
    for n in (8192, 262144, 1 << 20):
        by = {r["leg"]: r for r in result["rows"] if r["n_particles"] == n}
        result.setdefault("overhead_us", {})[str(n)] = {
            "p0_step": (by["p0"]["step_ms_median"] - by["off"]["step_ms_median"]) * 1e3,
            "p0_resample_phase": (by["p0"]["resample_phase_ms"] - by["off"]["resample_phase_ms"]) * 1e3,
            "p_high_resample_phase": (by["p_high"]["resample_phase_ms"] - by["off"]["resample_phase_ms"]) * 1e3}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result))


if __name__ == "__main__":
    main()
