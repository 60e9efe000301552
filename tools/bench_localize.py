"""Localiser benchmark on one B200: map load (term table) time for both sensor models at 1024^2 and 2048^2, the
per-step time of GridMapLocalizer at configs[2]'s scene (20 m room, 1024^2 at 5 cm, 6 m lidar, 360 beams, map from
scene_map) for 8,192 .. 1,048,576 particles, and two reference points measured in the same process: the SLAM step at
configs[2] and the CPU oracle localiser (one thread, bounded N). Writes profiles/loc_bench_1gpu.json (or --out).
Needs a GPU: there is no fallback.

    python tools/bench_localize.py [--steps 50] [--warmup 3] [--out profiles/loc_bench_1gpu.json]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from slamrs_b200 import GpuPlacement, GridMapLocalizer, GridMapSlam, SensorModel, grid_cells  # noqa: E402
from slamrs_b200.simulator import scene_map  # noqa: E402
from slamrs_b200.workloads import WORKLOADS  # noqa: E402

SEED = 0x5EED5A11
MODELS = {"beam_endpoint": SensorModel(), "likelihood_field": SensorModel.likelihood_field(sigma=0.1, z_rand=0.05)}


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True, check=True).stdout.strip().splitlines()[0]
    name, power = (s.strip() for s in out.split(","))
    return {"name": name, "power_limit": power}


def timed_steps(filt, odo, steps, warmup):
    """Median device time of one step_async over `steps` steps (CUDA events on the handle's stream)."""
    import torch
    stream = torch.cuda.ExternalStream(filt.stream_ptr)
    for _ in range(warmup):
        filt.step_async(odo)
    filt.sync()
    times = []
    for _ in range(steps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        filt.step_async(odo)
        b.record(stream)
        b.synchronize()
        times.append(a.elapsed_time(b))
    filt.sync()
    return float(np.median(times)), float(np.min(times)), float(np.max(times))


def map_load(grid, model):
    """Host clock around create: the map upload, the term table (and the distance transform) and allocation."""
    import torch
    res = 0.05
    w = grid * res
    from slamrs_b200 import GridMapSlamConfig
    cfg = GridMapSlamConfig(position=(-w / 2, -w / 2), width=w, height=w, resolution=res, n_particles=1024)
    scale = 10.0 if grid == 1024 else 20.0
    from slamrs_b200.simulator import reference_scene
    prob = scene_map(reference_scene(scale), cfg)
    out = []
    for _ in range(4):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        loc = GridMapLocalizer(cfg, prob, model, GpuPlacement(seed=SEED))
        t1 = time.perf_counter()
        loc.close()
        out.append((t1 - t0) * 1e3)
    return {"grid": grid, "create_ms_median_of_3": float(np.median(out[1:])), "first_create_ms": out[0]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "loc_bench_1gpu.json"))
    ap.add_argument("--cpu-particles", type=int, default=2048)
    args = ap.parse_args()
    import torch
    if torch.cuda.device_count() == 0:
        raise SystemExit("bench_localize: no GPU visible (the localiser has no CPU path)")
    result = {"card": card(), "steps": args.steps, "warmup": args.warmup, "map_load": {}, "step": {}}
    for name, model in MODELS.items():
        result["map_load"][name] = [map_load(g, model) for g in (1024, 2048)]

    wl = WORKLOADS["c3"]
    sim = wl.simulator()
    obs, odo = sim.next_scan(wl.speed_left, wl.speed_right)
    n_valid = int(obs.valid.sum())
    half = 0.9 * wl.scene_scale
    for name, model in MODELS.items():
        rows = []
        for n in (8192, 65536, 262144, 1 << 20):
            cfg = wl.slam_config(n)
            with GridMapLocalizer(cfg, scene_map(sim.segments, cfg), model, GpuPlacement(seed=SEED)) as loc:
                loc.init_uniform((-half, -half, half, half))
                loc.upload_scan(obs)
                med, lo, hi = timed_steps(loc, odo, args.steps, args.warmup)
                before = loc.launch_count
                loc.step_async(odo)
                launches = loc.launch_count - before
                loc.set_profiling(True)
                for _ in range(args.steps):
                    loc.step_async(odo)
                ms, k = loc.phase_ms()
                loc.set_profiling(False)
            rows.append({"n_particles": n, "step_ms_median": med, "step_ms_min": lo, "step_ms_max": hi,
                         "particle_beam_evals_per_s": n * n_valid / (med * 1e-3), "launches_per_step_async": launches,
                         "k_loc_step_ms": ms["motion_likelihood"] / k, "weights_and_indices_ms": ms["resample"] / k})
            print(name, rows[-1], flush=True)
        result["step"][name] = rows
    result["valid_beams"] = n_valid

    # reference point 1: the SLAM step at configs[2] (8,192 particles), same scan, same process
    with GridMapSlam(wl.slam_config(), GpuPlacement(seed=SEED)) as slam:
        slam.upload_scan(obs)
        med, lo, hi = timed_steps(slam, odo, args.steps, args.warmup)
    result["slam_step_c3"] = {"n_particles": wl.n_particles, "step_ms_median": med, "step_ms_min": lo, "step_ms_max": hi}

    # reference point 2: the CPU oracle localiser, one thread, bounded N (the CPU baseline)
    from oracle import loc_oracle as LO
    from oracle import oracle as O
    n = args.cpu_particles
    cfg = wl.slam_config(n)
    g = grid_cells(cfg.width, cfg.resolution)
    cpu = {}
    for name, model in MODELS.items():
        ol = LO.OracleLocalizer(cfg.position, cfg.resolution, g, g, n, scene_map(sim.segments, cfg), model.kind, model.sigma,
                               model.z_rand, model.occupied_above)
        ol.set_poses(O.uniform_poses(SEED, 0, n, (-half, -half, half, half)))
        ang = obs.angle.astype(np.float32).astype(np.float64)
        dist = obs.distance.astype(np.float32).astype(np.float64)
        ts = []
        for step in range(3):
            z = O.motion_normals(SEED, step, 0, n)
            t0 = time.perf_counter()
            ol.update(ang, dist, obs.valid.astype(np.uint8), np.float32(odo.distance_left), np.float32(odo.distance_right),
                      np.float32(odo.wheel_distance), z, O.resample_uniform(SEED, step))
            ts.append((time.perf_counter() - t0) * 1e3)
        ol.close()
        cpu[name] = {"n_particles": n, "step_ms_median": float(np.median(ts)),
                     "particle_beam_evals_per_s": n * n_valid / (np.median(ts) * 1e-3)}
    result["cpu_oracle_single_thread"] = cpu
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result))


if __name__ == "__main__":
    main()
