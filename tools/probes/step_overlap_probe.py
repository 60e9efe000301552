#!/usr/bin/env python
"""A/B probe of the step chain: ms per step of bench.py's `value` loop (configs[2] by default, device-resident scans,
step_async back to back, no host synchronisation inside the timed window) with per-phase profiling off and on, and
with SLAMRS_FLAG_SERIAL_STEPS (the serial kernel sequence with stream events between the phases) off and on. Legs
alternate inside one process, `--rounds` times each, on one filter per leg over the same seeded scans.

    python tools/probes/step_overlap_probe.py [--steps 64] [--warmup 8] [--rounds 3] [--workload c3] [--particles N]
    python tools/probes/step_overlap_probe.py --libs A.so B.so   # alternate two builds of the library, one process each

Prints the card name, power limit and SM clocks, then one JSON line per leg and round, then the median per leg."""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)


def card_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        out = ""
    return dict(zip(q.split(","), [s.strip() for s in out.split(",")])) if out else {}


def run_legs(args):
    import numpy as np
    import torch
    from slamrs_b200 import GpuPlacement, GridMapSlam, _lib
    from slamrs_b200.workloads import WORKLOADS

    if not torch.cuda.is_available():
        raise SystemExit("step_overlap_probe: no CUDA device")
    dev = torch.device("cuda", 0)
    wl = WORKLOADS[args.workload]
    if args.particles:
        wl = wl.__class__(**{**wl.__dict__, "n_particles": args.particles})
    K, W = args.steps, args.warmup
    sim = wl.simulator()
    scans = [sim.next_scan(wl.speed_left, wl.speed_right) for _ in range(W + K)]
    d_scans = []
    for obs, odo in scans:
        d_scans.append((torch.from_numpy(obs.angle.astype(np.float32)).to(dev),
                        torch.from_numpy(obs.distance.astype(np.float32)).to(dev),
                        torch.from_numpy(obs.valid.astype(np.uint8)).to(dev),
                        float(obs.distance.max()) if len(obs) else 0.0, odo))
    torch.cuda.synchronize()

    def leg(serial, profiling):
        flags = _lib.FLAG_SERIAL_STEPS if serial else 0
        slam = GridMapSlam(wl.slam_config(wl.n_particles), GpuPlacement(device=0, flags=flags, slot_cells=wl.slot_cells))
        if wl.uniform_init:
            from slamrs_b200.workloads import uniform_poses
            slam.set_poses(uniform_poses(wl, slam.first, slam.n_local))
        stream = torch.cuda.ExternalStream(slam.stream_ptr, device=dev)

        def step(i):
            a, d, v, maxd, odo = d_scans[i]
            slam.set_scan_device(a.data_ptr(), d.data_ptr(), v.data_ptr(), a.numel(), maxd)
            slam.step_async(odo)
        for i in range(W):
            step(i)
        slam.sync()
        slam.set_profiling(profiling)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record(stream)
        for i in range(W, W + K):
            step(i)
        e1.record(stream)
        slam.sync()
        ms = e0.elapsed_time(e1) / K
        phases = None
        if profiling:
            ph, n = slam.phase_ms()
            phases = {k: round(v / max(n, 1), 5) for k, v in ph.items()}
        w = slam.weights()
        digest = float(np.asarray(w[0] if isinstance(w, tuple) else w, dtype=np.float64).sum())
        slam.close()
        return ms, phases, digest

    legs = [(s, p) for s in (False, True) for p in (False, True)]
    series = {}
    for r in range(args.rounds):
        for serial, prof in legs:
            ms, phases, digest = leg(serial, prof)
            name = f"{'serial' if serial else 'default'}_prof_{'on' if prof else 'off'}"
            series.setdefault(name, []).append(ms)
            print(json.dumps({"lib": args.lib_name, "round": r, "leg": name, "ms_per_step": round(ms, 5),
                              "phases_ms_per_step": phases, "weight_sum": digest}), flush=True)
    for name, v in series.items():
        print(json.dumps({"lib": args.lib_name, "leg": name, "median_ms_per_step": round(statistics.median(v), 5),
                          "min": round(min(v), 5), "max": round(max(v), 5)}), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=64)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--workload", default="c3")
    ap.add_argument("--particles", type=int, default=0)
    ap.add_argument("--libs", nargs="*", default=None, help="library builds to alternate (one process per build and round)")
    ap.add_argument("--lib-name", default="tree", help=argparse.SUPPRESS)
    args = ap.parse_args()
    print(json.dumps({"card": card_info()}), flush=True)
    if not args.libs:
        run_legs(args)
        return
    for r in range(args.rounds):
        for lib in args.libs:
            cmd = [sys.executable, os.path.abspath(__file__), "--steps", str(args.steps), "--warmup", str(args.warmup),
                   "--rounds", "1", "--workload", args.workload, "--particles", str(args.particles),
                   "--lib-name", os.path.basename(lib)]
            env = dict(os.environ, SLAMRS_GPU_LIB=os.path.abspath(lib))
            subprocess.run(cmd, env=env, check=True)


if __name__ == "__main__":
    main()
