"""Cost of the localiser's pose clusters (slamrs_gpu_pose_clusters) on one B200.

For 8,192, 262,144 and 1,048,576 poses on the at-scale map (512^2 at 5 cm), once for a converged cloud (every pose
within a few centimetres and degrees of one pose) and once for a uniform one (init_uniform over the whole map), with
Clustering() (0.5 m / 10 degree bins, 16 clusters): the median device time of the call (CUDA events around it on the
handle's stream) and the median host time of the synchronous call, over --calls calls after --warmup, next to the
device time of one localiser step at the same population (likelihood field, 360 beams). Card and power limit are read
in the same run. Writes profiles/loc_clusters_1gpu.json (or --out). Needs a GPU.

    python tools/bench_loc_clusters.py [--calls 50] [--warmup 10] [--out profiles/loc_clusters_1gpu.json]
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_localize import card, timed_steps  # noqa: E402
from common import at_scale_config, make_scans  # noqa: E402
from slamrs_b200 import Clustering, GpuPlacement, GridMapLocalizer, SensorModel  # noqa: E402
from slamrs_b200.simulator import reference_scene, scene_map  # noqa: E402

SEED = 0x5EED5A11
MODEL = SensorModel.likelihood_field(sigma=0.1, z_rand=0.05)


def measure(n, cloud, calls, warmup):
    import torch
    cfg = at_scale_config(n)
    obs, odo = make_scans(10.0, 360, 6.0, 1)[0]
    cl = Clustering()
    with GridMapLocalizer(cfg, scene_map(reference_scene(10.0), cfg), MODEL, GpuPlacement(seed=SEED)) as loc:
        if cloud == "converged":
            rng = np.random.default_rng(n)
            loc.set_poses(np.column_stack([rng.normal(1.0, 0.03, n), rng.normal(-0.5, 0.03, n),
                                           rng.normal(0.4, 0.02, n)]).astype(np.float32))
        else:
            loc.init_uniform((-12.8, -12.8, 12.8, 12.8))
        stream = torch.cuda.ExternalStream(loc.stream_ptr)
        for _ in range(warmup):
            overall, clusters = loc.pose_clusters(cl)
        dev, host = [], []
        for _ in range(calls):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            t0 = time.perf_counter()
            loc.pose_clusters(cl)
            host.append((time.perf_counter() - t0) * 1e3)
            b.record(stream)
            b.synchronize()
            dev.append(a.elapsed_time(b))
        loc.upload_scan(obs)
        step_ms = timed_steps(loc, odo, calls, warmup)
    return {"n": n, "cloud": cloud, "n_bins": overall["n_bins"], "n_clusters": overall["n_clusters"],
            "call_device_ms_median": statistics.median(dev), "call_device_ms_min": min(dev),
            "call_host_ms_median": statistics.median(host), "step_device_ms_median": step_ms[0]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "loc_clusters_1gpu.json"))
    args = ap.parse_args()
    rows = [measure(n, cloud, args.calls, args.warmup) for n in (8192, 262144, 1 << 20) for cloud in ("converged", "uniform")]
    result = {"card": card(), "calls": args.calls, "warmup": args.warmup, "clustering": "Clustering()", "rows": rows}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result))


if __name__ == "__main__":
    main()
