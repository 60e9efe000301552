"""Cost of scan-matching pose refinement on one B200: configs[2]'s scene (20 m room, 1024^2 grid at 5 cm, 6 m lidar,
360 beams) at 256, 1,024 and 8,192 particles, with the matcher off and on (ScanMatcher() defaults). For each, the
median over steps 30-80 (the map has content by then) of the step time (CUDA events on the handle's stream) and of the
MOTION_LIKELIHOOD phase (where k_scan_match is accounted, from a second run with phase profiling on), and the
per-step scan-match statistics. Writes profiles/scan_match_1gpu.json (or --out). Needs a GPU: there is no fallback.

    python tools/bench_scan_match.py [--sizes 256,1024,8192] [--out profiles/scan_match_1gpu.json]
"""
from __future__ import annotations

import argparse
import dataclasses
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from slamrs_b200 import GpuPlacement, GridMapSlam, ScanMatcher  # noqa: E402
from slamrs_b200.workloads import WORKLOADS  # noqa: E402

SEED = 0x5EED5A11
FIRST, LAST = 30, 80   # the timed window, steps FIRST .. LAST inclusive


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True, check=True).stdout.strip().splitlines()[0]
    name, power = (s.strip() for s in out.split(","))
    return {"name": name, "power_limit": power}


def run(n, matcher, scans, profile):
    """Per step: device ms (or motion_likelihood phase ms with profile) and scan-match stats."""
    import torch
    wl = WORKLOADS["c3"]
    times, stats = [], []
    with GridMapSlam(wl.slam_config(n), GpuPlacement(seed=SEED)) as g:
        g.set_scan_matcher(matcher)
        stream = torch.cuda.ExternalStream(g.stream_ptr)
        if profile:
            g.set_profiling(True)
        for step, (obs, odo) in enumerate(scans):
            g.upload_scan(obs)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            g.step_async(odo)
            b.record(stream)
            b.synchronize()
            if profile:
                ph, _ = g.phase_ms()
                times.append(ph["motion_likelihood"])
            else:
                times.append(a.elapsed_time(b))
            st = g.scan_match_stats()
            stats.append([st["moved"], st["moves"], st["scored"], st["capped"]])
    return np.array(times[FIRST:LAST + 1]), np.array(stats[FIRST:LAST + 1])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="256,1024,8192")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "scan_match_1gpu.json"))
    args = ap.parse_args()
    wl = WORKLOADS["c3"]
    sim = wl.simulator()
    scans = [sim.next_scan(wl.speed_left, wl.speed_right) for _ in range(LAST + 1)]
    result = {"card": card(), "workload": wl.name, "matcher": dataclasses.asdict(ScanMatcher()),
              "window": [FIRST, LAST], "rows": []}
    for n in (int(s) for s in args.sizes.split(",")):
        for label, m in (("off", None), ("on", ScanMatcher())):
            t, st = run(n, m, scans, profile=False)
            ph, _ = run(n, m, scans, profile=True)
            row = {"n_particles": n, "matcher": label, "step_ms_median": float(np.median(t)),
                   "step_ms_min": float(t.min()), "step_ms_max": float(t.max()),
                   "motion_likelihood_ms_median": float(np.median(ph)),
                   "stats_per_step_median": dict(zip(("moved", "moves", "scored", "capped"),
                                                     (float(v) for v in np.median(st, axis=0)))),
                   "scored_per_particle_mean": float(st[:, 2].mean() / n)}
            result["rows"].append(row)
            print(json.dumps(row), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result["card"]))


if __name__ == "__main__":
    main()
