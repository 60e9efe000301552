"""Cost and behaviour of the localiser's KLD-sampling (adaptive population, slamrs_gpu_set_kld) on one B200.

(a) machinery   configs[2]'s scene (20 m room, 1024^2 at 5 cm, free space marked, 6 m lidar, 360 beams, likelihood
                field), robot standing still, particles at the true pose, for 8,192, 262,144 and 1,048,576 particles:
                KLD-sampling off against on at a fixed population (n_min = n_max = n, so both legs weight and draw the
                same n). Device time per step (CUDA events around step_async), host time of update() (scan upload,
                step, synchronise) and host time per step of a loop of step_async calls (the host now waits for
                k_loc_kld's bin count inside step_async).
(b) global      the scene and seed of test_global_localisation_from_a_uniform_start (10 m room, 512^2 at 5 cm, 2^20
                particles from a uniform start), 40 scans with Kld() beside the fixed 2^20 run: population, k,
                device step time and error per scan.
(c) kidnapped   the kidnapped-robot scenario of DESIGN.md section 11.1 (carried to (3.5, 3.0) and turned by 2 rad after
                scan 20) with Kld() and Recovery(): population and injections per scan, and whether the population
                grows after the first injection.

Card and power limit are read in the same run. Writes profiles/loc_kld_1gpu.json (or --out). Needs a GPU.

    python tools/bench_loc_kld.py [--steps 50] [--warmup 5] [--out profiles/loc_kld_1gpu.json]
"""
from __future__ import annotations

import argparse
import json
import math
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_localize import card  # noqa: E402
from common import at_scale_config  # noqa: E402
from slamrs_b200 import GpuPlacement, GridMapLocalizer, Kld, Odometry, Recovery, SensorModel  # noqa: E402
from slamrs_b200.simulator import Simulator, reference_scene, scene_map  # noqa: E402
from slamrs_b200.workloads import WORKLOADS  # noqa: E402
from test_gpu_localize_kld import room_map  # noqa: E402

SEED = 0x5EED5A11
MODEL = SensorModel.likelihood_field(sigma=0.1, z_rand=0.05)


def _events():
    import torch
    return torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)


def machinery(steps, warmup):
    import torch
    wl = WORKLOADS["c3"]
    sim = wl.simulator()
    obs, _ = sim.next_scan(wl.speed_left, wl.speed_right)
    odo = Odometry(0.0, 0.0, wl.wheel_base)
    truth = np.array([[float(v) for v in sim.pose]], np.float32)
    rows = []
    for n in (8192, 262144, 1 << 20):
        cfg = wl.slam_config(n)
        prob = room_map(sim.segments, cfg)
        for leg in ("off", "fixed"):
            with GridMapLocalizer(cfg, prob, MODEL, GpuPlacement(seed=SEED)) as loc:
                loc.set_kld(None if leg == "off" else Kld(n_min=n, n_max=n))
                loc.set_poses(np.repeat(truth, n, axis=0))
                loc.upload_scan(obs)
                stream = torch.cuda.ExternalStream(loc.stream_ptr)
                for _ in range(warmup):
                    loc.step_async(odo)
                loc.sync()
                dev = []
                for _ in range(steps):
                    a, b = _events()
                    a.record(stream)
                    loc.step_async(odo)
                    b.record(stream)
                    b.synchronize()
                    dev.append(a.elapsed_time(b))
                upd = []
                for _ in range(steps):
                    t0 = time.perf_counter()
                    loc.update(obs, odo)
                    upd.append((time.perf_counter() - t0) * 1e3)
                loc.sync()
                t0 = time.perf_counter()
                for _ in range(steps):
                    loc.step_async(odo)
                loc.sync()
                loop = (time.perf_counter() - t0) * 1e3 / steps
                st = loc.kld_state()
                assert loc.population == n
            row = {"n_particles": n, "leg": leg, "device_step_ms_median": float(np.median(dev)),
                   "device_step_ms_min": float(np.min(dev)), "device_step_ms_max": float(np.max(dev)),
                   "host_update_ms_median": float(np.median(upd)), "host_step_async_loop_ms_per_step": loop,
                   "k_last": st["k"]}
            rows.append(row)
            print(row, flush=True)
    over = {}
    for n in (8192, 262144, 1 << 20):
        by = {r["leg"]: r for r in rows if r["n_particles"] == n}
        over[str(n)] = {k: (by["fixed"][k] - by["off"][k]) * 1e3 for k in
                        ("device_step_ms_median", "host_update_ms_median", "host_step_async_loop_ms_per_step")}
    return {"workload": "c3 scene, likelihood field, particles at the true pose, robot still", "rows": rows,
            "overhead_us": over}


def _run(kld, recovery=None, kidnap=False, scans=40):
    import torch
    cfg = at_scale_config(1 << 20)
    segments = reference_scene(5.0)
    sim = Simulator(segments, n_beams=360, scanner_range=6.0, wheel_base=0.1)
    prob = room_map(segments, cfg) if recovery is not None else scene_map(segments, cfg)
    trace = []
    with GridMapLocalizer(cfg, prob, MODEL, GpuPlacement(seed=SEED)) as loc:
        loc.set_kld(kld)
        loc.set_recovery(recovery)
        loc.init_uniform((-4.5, -4.5, 4.5, 4.5))
        stream = torch.cuda.ExternalStream(loc.stream_ptr)
        for s in range(scans):
            if kidnap and s == 20:
                t = float(sim.pose[2])
                sim.pose = [np.float32(3.5), np.float32(3.0), np.float32(t + 2.0)]
            obs, odo = sim.next_scan(0.08, 0.10)
            n_t = loc.population
            loc.upload_scan(obs)
            a, b = _events()
            a.record(stream)
            loc.step_async(odo)
            b.record(stream)
            b.synchronize()
            ep = loc.estimated_pose()
            row = {"scan": s, "n_weighted": n_t, "k": loc.kld_state()["k"], "n_drawn": loc.population,
                   "step_ms": round(a.elapsed_time(b), 4),
                   "err_m": round(math.hypot(ep.x - float(sim.pose[0]), ep.y - float(sim.pose[1])), 4),
                   "err_rad": round(abs(math.remainder(ep.theta - float(sim.pose[2]), 2.0 * math.pi)), 4)}
            if recovery is not None:
                row["injected"] = loc.recovery_state()["injected"]
            trace.append(row)
            print(row, flush=True)
    return trace


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "loc_kld_1gpu.json"))
    args = ap.parse_args()
    import torch
    if torch.cuda.device_count() == 0:
        raise SystemExit("bench_loc_kld: no GPU visible (the localiser has no CPU path)")
    result = {"card": card(), "steps": args.steps, "warmup": args.warmup}
    result["a_machinery"] = machinery(args.steps, args.warmup)
    result["b_global"] = {"kld": _run(Kld()), "fixed": _run(None)}
    kid = _run(Kld(), Recovery(), kidnap=True, scans=60)
    first = next((r["scan"] for r in kid if r.get("injected", 0) > 0), None)
    grows = None if first is None else any(r["n_drawn"] > kid[first]["n_weighted"] for r in kid[first:])
    result["c_kidnapped"] = {"trace": kid, "first_injection_scan": first, "population_grows_after_injection": grows}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps({k: v for k, v in result.items() if k != "b_global" and k != "c_kidnapped"}))
    print("kidnapped: first injection", first, "population grows after it:", grows)


if __name__ == "__main__":
    main()
