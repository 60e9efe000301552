#!/usr/bin/env python
"""Benchmark of the grid particle-filter SLAM step (BASELINE.json metric: particle-beam updates/s,
plus the fraction of the measured HBM roofline reached by the dominant kernel).

    python bench.py --gpus N --steps K --warmup W              # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...    # the reference's CPU path (oracle port)

A "step" is one full GridMapSlam::update (slamrs/slam/src/grid/slam.rs:46-75) over one synthetic
simulator scan: motion sample + beam likelihood + ray update for every particle, weight
normalisation, systematic resampling, grid copies. Workload at N GPUs = N shards of configs[2]
(8,192 particles x 360 beams on a 1024^2 grid per GPU; 8 GPUs = configs[3], 65,536 particles),
i.e. weak scaling. Under torchrun each rank drives one GPU; rank 0 prints ONE JSON line.

Legs of the CUDA arm
  value  K steps on device-resident scans, no host synchronisation inside the timed region,
         CUDA events on the library's stream, max over ranks.
  e2e    K steps through the reference-facing call sequence of GridMapSlamNode::update
         (node.rs:47-60): update(host scan) -> estimated_pose() -> estimated_likelihood() into a
         pinned host grid; host<->device copies inside the timed region. `e2e` runs the read-out
         pipelined by one step (estimated_likelihood_async + map_wait: map t is copied while
         update(t+1) runs), `e2e_blocking` with every call blocking.
  roofline  the kernel that takes most of the step. With deferred copies (default) that is the ray
         update: 8 B per step of the reference's ray iterator (SURVEY.md 8(d)), steps counted by the
         kernel, over the kernel's own CUDA-event time, against MEASURED_PEAKS.json's HBM copy
         bandwidth. roofline_copy is the same for the copy kernels (bytes really read + written,
         counted on the device: whole tiles of the informed extent of every grid written and read).
  eager_copy / full_grid_copy / strict_order_of_work  the same run with every clone copied when
         resampling creates it (extent copies), with whole-grid copies (what Map::clone moves) and
         with the reference's order of work; results are identical in all modes.
  cpu_baseline  (N=1, rank 0) the CPU oracle on a bounded sample of the same workload.

--dump-outputs DIR writes what the `value` leg's filter holds after its last timed step (resample indices, argmax,
normalised weights, all poses, published pose and map; see step_outputs) as DIR/<name>.npy. Scans and random draws
are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "particle_beam_updates_per_s"
UNIT = "particle-beam updates/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=16)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["cuda", "reference"], default="cuda")
    ap.add_argument("--workload", default="c3", help="c1 | c2 | c3 | c5 (per-GPU shard; default configs[2])")
    ap.add_argument("--particles", type=int, default=0, help="override particles per GPU")
    ap.add_argument("--cpu-particles", type=int, default=0, help="particles of the bounded CPU sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-strict", action="store_true", help="skip the strict-order-of-work comparison run")
    ap.add_argument("--no-full-copy", action="store_true", help="skip the whole-grid-copy comparison run")
    ap.add_argument("--no-eager", action="store_true", help="skip the eager-copy comparison run")
    ap.add_argument("--no-aged", action="store_true", help="skip the aged-map leg (timed steps after 160 more scans)")
    ap.add_argument("--no-c5", action="store_true", help="skip the configs[4] leg of an 8-GPU run")
    ap.add_argument("--c5-leg", action="store_true", help="run the configs[4] shard leg at any GPU count")
    ap.add_argument("--flags", type=int, default=0, help="slamrs_flags bits for the main run (profiling)")
    ap.add_argument("--shift-x-cells", type=int, default=0, help="experiment: move the map origin by this many cells in x")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed path computed in its last step as DIR/<name>.npy (CUDA arm)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "cuda":
        ap.error("--dump-outputs writes the outputs of the CUDA arm")
    return args


# ------------------------------------------------------------------------------ helpers
def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled every 200 ms while the timed region runs."""
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
              "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu_index = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.gpu_index}", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                 "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, smax, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            p = [x.strip() for x in ln.split(",")]
            if len(p) < 9:
                continue
            try:
                sm.append(float(p[1])); smax.append(float(p[2])); power.append(float(p[3]))
            except ValueError:
                continue
            for name, v in zip(names, p[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        # "under load": samples in the upper half of the observed power range
        pw = np.array(power); smv = np.array(sm)
        load = smv[pw >= (pw.min() + pw.max()) / 2.0] if pw.max() > pw.min() else smv
        return {"sm_mhz": float(np.median(load)), "sm_max_mhz": float(max(smax)), "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": float(pw.max())}


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


# ------------------------------------------------------------------------------ reference arm
def run_reference(args, wl, rank, world):
    """The reference's own CPU implementation of the path: the C oracle (a port -- the Rust
    reference cannot be compiled in this image), all host threads, bounded sample per step."""
    if rank != 0:
        return  # rank 0 alone runs the CPU arm
    from oracle import oracle as O
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    cores = os.cpu_count() or 1
    n_cpu = args.cpu_particles or max(cores * 8, 64)
    res = time_oracle(O, wl, n_cpu, args.steps, args.warmup, cores)
    line = {
        "impl": "reference", "metric": METRIC, "value": res["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": res["ms_per_step"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32 geometry, f64 cells/weights", "data": "synthetic",
        "config": workload_config(wl, args.gpus, wl.n_particles * args.gpus),
        "cpu_baseline": {"value": res["value"], "unit": UNIT, "cores": cores, "kind": "port", "sample": res["sample"]},
        "e2e": {"value": res["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def time_oracle(O, wl, n_cpu, steps, warmup, threads, dead_likelihood=False):
    from slamrs_b200.slam import GridMapSlamConfig  # noqa: F401  (host types only)
    cfg = wl.slam_config(n_cpu)
    sim = wl.simulator()
    scans = [sim.next_scan(wl.speed_left, wl.speed_right) for _ in range(warmup + steps)]
    osl = O.OracleSlam(cfg.position, cfg.width, cfg.height, cfg.resolution, n_cpu, False)
    osl.set_threads(threads)
    osl.set_dead_likelihood(dead_likelihood)
    seed = 0x5EED5A11
    times = []
    for s, (obs, odo) in enumerate(scans):
        z = O.motion_normals(seed, s, 0, n_cpu)
        u = O.resample_uniform(seed, s)
        ang = obs.angle.astype(np.float32).astype(np.float64)
        dist = obs.distance.astype(np.float32).astype(np.float64)
        t0 = time.perf_counter()
        osl.update(ang, dist, obs.valid.astype(np.uint8), np.float32(odo.distance_left),
                   np.float32(odo.distance_right), np.float32(odo.wheel_distance), z, u)
        osl.estimated_pose(); osl.estimated_likelihood()   # what the node publishes per scan (node.rs:51-57)
        dt = time.perf_counter() - t0
        if s >= warmup:
            times.append(dt)
    osl.close()
    total = float(sum(times))
    return {"value": n_cpu * wl.n_beams * len(times) / total, "ms_per_step": 1e3 * total / len(times),
            "sample": f"{n_cpu} particles x {wl.n_beams} beams, {wl.grid}^2 f64 grid, {len(times)} steps after "
                      f"{warmup} warm-up, {threads} OpenMP threads over particles"
                      f"{', with the dead Map::likelihood() transform' if dead_likelihood else ''}"}


def workload_config(wl, n_gpus, n_total):
    return {"workload": f"{n_total} particles x {wl.n_beams} beams, {wl.grid}x{wl.grid} grid @ {wl.resolution} m "
                        f"({wl.name} shard per GPU; simulator scene x{wl.scene_scale:g}, range {wl.scanner_range:g} m)",
            "particles_per_gpu": wl.n_particles, "beams": wl.n_beams, "grid": wl.grid, "slot_cells": wl.slot_cells,
            "parallelism": f"particles sharded dp{n_gpus}",
            "l2": "working set (per-particle grids) is far larger than L2; no flush needed"}


# ------------------------------------------------------------------------------ CUDA arm
def step_outputs(slam, world, dev):
    """What a caller holds after a step: the resample index vector, the argmax, the normalised weights, the poses of
    the whole population, the published pose and the published map (row-major, grid_w x grid_h)."""
    import torch
    import torch.distributed as dist
    poses = torch.from_numpy(slam.poses()).to(dev)
    if world > 1:
        parts = [torch.empty_like(poses) for _ in range(world)]
        dist.all_gather(parts, poses)
        poses = torch.cat(parts)
    ep = slam.estimated_pose()
    m = slam.estimated_likelihood().data          # collective: every rank reads the owner's grid
    return {"resample_indices": slam.resample_indices(), "max_particle": np.array([slam.max_particle], np.uint64),
            "weights": slam.weights()[0], "poses": poses.cpu().numpy(),
            "estimated_pose": np.array([ep.x, ep.y, ep.theta], np.float32),
            "estimated_likelihood": m.reshape(slam.grid_w, slam.grid_h)}


def state_hash(outputs):
    """SHA-256 over what a step leaves behind (step_outputs without the weights). Equal hashes = identical filter
    state."""
    import hashlib
    h = hashlib.sha256()
    for name in ("resample_indices", "max_particle", "poses", "estimated_pose", "estimated_likelihood"):
        h.update(outputs[name].tobytes())
    return h.hexdigest()


DUMP_BYTES = 64_000_000


def dump_outputs(path, outputs):
    """Writes every output as <path>/<name>.npy: float32 stays float32, everything else becomes float64 (indices
    and counts are exact below 2**53). All files together hold at most 64 MB: an output larger than its share is
    replaced by a fixed, seeded sample of its elements, so that two runs still compare element for element."""
    os.makedirs(path, exist_ok=True)
    items = sorted(outputs.items(), key=lambda kv: kv[1].nbytes)
    left = DUMP_BYTES - 4096 * len(items)         # room for the .npy headers
    for i, (name, a) in enumerate(items):
        a = a.astype(np.float32 if a.dtype == np.float32 else np.float64)
        share = left // (len(items) - i)
        if a.nbytes > share:
            keep = np.random.default_rng(0).choice(a.size, share // a.itemsize, replace=False)
            a = a.reshape(-1)[np.sort(keep)]
        np.save(os.path.join(path, name + ".npy"), a)
        left -= a.nbytes


STEP_HISTORY = 256   # per-step records the library keeps (include/slamrs_gpu.h)


def step_history(slam, first, count):
    """The per-step records of steps first .. first+count-1 as float64. A run longer than the library's ring
    repeats the records of its last STEP_HISTORY steps, so that sums over the rows still stand for `count` steps."""
    n = min(count, STEP_HISTORY)
    hist = slam.step_history(first + count - n, n).astype(np.float64)
    return np.resize(hist, (count, hist.shape[1]))


def measure_e2e_pipelined(args, wl, rank, world, local, dev, nccl_id, scans, flags):
    """The headline end-to-end leg on a filter of its own and on the SAME scans as the device-resident `value` leg
    (W warm-up scans, then K timed ones): update(host scan) -> estimated_pose() -> the 8 B/cell map into page-locked
    host memory every step, the map copy of step t overlapping update(t+1). Returns elapsed ms (CUDA events on the
    library's stream, recorded around host-synchronised work)."""
    import torch
    import torch.distributed as dist
    from slamrs_b200 import GpuPlacement, GridMapSlam

    K, W = args.steps, args.warmup
    cfg = wl.slam_config(wl.n_particles * world)
    slam = GridMapSlam(cfg, GpuPlacement(device=local, rank=rank, world_size=world, nccl_id=nccl_id, flags=flags,
                                         slot_cells=wl.slot_cells))
    if wl.uniform_init:
        from slamrs_b200.workloads import uniform_poses
        slam.set_poses(uniform_poses(wl, slam.first, slam.n_local))
    stream = torch.cuda.ExternalStream(slam.stream_ptr, device=dev)
    bufs = [torch.empty(slam.grid_w * slam.grid_h, dtype=torch.float64).pin_memory().numpy() for _ in range(2)]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step(i, obs, odo):
        slam.update(obs, odo)                  # GridMapSlam::update with HOST scan buffers (blocks until the step is done)
        slam.estimated_pose()                  # node.rs:51
        slam.map_wait()                        # map i-1 has landed (it was copied while step i ran): publish it
        slam.estimated_likelihood_async(bufs[i & 1] if rank == 0 else None)   # node.rs:53-57, pipelined by one step

    for i, (obs, odo) in enumerate(scans[:W]):
        step(i, obs, odo)
    slam.map_wait()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record(stream)
    for i, (obs, odo) in enumerate(scans[W:W + K]):
        step(i, obs, odo)
    slam.map_wait()
    e1.record(stream)
    slam.sync()
    barrier()
    ms = e0.elapsed_time(e1)
    slam.close()
    return ms


def measure_cuda(args, wl, rank, world, local, dev, nccl_id, scans, flags, do_e2e, do_aged=False):
    """One filter run: W warm-up + K timed device-resident steps (+ K e2e steps). Returns a dict of
    rank-local measurements; the caller reduces over ranks."""
    import torch
    import torch.distributed as dist
    from slamrs_b200 import GpuPlacement, GridMapSlam

    K, W = args.steps, args.warmup
    n_total = wl.n_particles * world
    cfg = wl.slam_config(n_total)
    if getattr(args, "shift_x_cells", 0):
        cfg.position = (cfg.position[0] - args.shift_x_cells * cfg.resolution, cfg.position[1])
    slam = GridMapSlam(cfg, GpuPlacement(device=local, rank=rank, world_size=world, nccl_id=nccl_id, flags=flags,
                                         slot_cells=wl.slot_cells))
    if wl.uniform_init:
        from slamrs_b200.workloads import uniform_poses
        slam.set_poses(uniform_poses(wl, slam.first, slam.n_local))
    stream = torch.cuda.ExternalStream(slam.stream_ptr, device=dev)
    grid_bytes = slam.stats()["bytes_per_grid"]

    d_scans = []
    for obs, odo in scans[:W + K]:
        a = torch.from_numpy(obs.angle.astype(np.float32)).to(dev)
        d = torch.from_numpy(obs.distance.astype(np.float32)).to(dev)
        v = torch.from_numpy(obs.valid.astype(np.uint8)).to(dev)
        d_scans.append((a, d, v, float(obs.distance.max()) if len(obs) else 0.0, odo))
    torch.cuda.synchronize()

    def device_step(i):
        a, d, v, maxd, odo = d_scans[i]
        slam.set_scan_device(a.data_ptr(), d.data_ptr(), v.data_ptr(), a.numel(), maxd)
        slam.step_async(odo)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(W):
        device_step(i)
    slam.sync()

    slam.set_profiling(True)
    launches0 = slam.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record(stream)
    for i in range(W, W + K):
        device_step(i)
    e1.record(stream)
    slam.sync()
    barrier()
    out = {"ms_value": e0.elapsed_time(e1), "launches": slam.launch_count - launches0, "grid_bytes": grid_bytes}
    out["phase_ms"], _ = slam.phase_ms()
    slam.set_profiling(False)
    out["hist"] = step_history(slam, W, K)
    out["stats"] = slam.stats()
    out["grid"] = (slam.grid_w, slam.grid_h)
    out["outputs"] = step_outputs(slam, world, dev)
    out["state_sha256"] = state_hash(out["outputs"])

    if do_e2e:
        pinned = torch.empty(slam.grid_w * slam.grid_h, dtype=torch.float64).pin_memory()
        out_np = pinned.numpy()
        barrier()
        e0.record(stream)
        for obs, odo in scans[W + K:W + 2 * K]:
            slam.update(obs, odo)                  # GridMapSlam::update with HOST scan buffers
            slam.estimated_pose()                  # node.rs:51
            if rank == 0:
                slam.estimated_likelihood(out_np)  # node.rs:53-57, 8 B/cell map into pinned host memory
            else:
                slam.skip_estimated_likelihood()   # one consumer (the node); the other ranks only take part
        e1.record(stream)
        slam.sync()
        barrier()
        out["ms_e2e_sync"] = e0.elapsed_time(e1)
        # the same loop with the cheaper read-out a visualizer needs: informed window only, f32
        pinned32 = torch.empty(slam.grid_w * slam.grid_h, dtype=torch.float32).pin_memory().numpy()
        barrier()
        e0.record(stream)
        win_bytes = 0
        for obs, odo in scans[W + 2 * K:W + 3 * K]:   # the trajectory continues: fresh scans
            slam.update(obs, odo)
            slam.estimated_pose()
            if rank == 0:
                _, w = slam.estimated_likelihood_window(out=pinned32)
                win_bytes += w.nbytes
            else:
                slam.skip_estimated_likelihood_window()
        e1.record(stream)
        slam.sync()
        barrier()
        out["ms_e2e_window"] = e0.elapsed_time(e1)
        out["e2e_window_bytes"] = win_bytes / max(1, K)
    if do_aged:
        # the same filter after AGED more scans: informed extents and survivor counts have grown
        base = W + 3 * K if do_e2e else W + K
        n_more = len(scans) - base - K
        d_more = []
        for obs, odo in scans[base:]:
            a = torch.from_numpy(obs.angle.astype(np.float32)).to(dev)
            d = torch.from_numpy(obs.distance.astype(np.float32)).to(dev)
            v = torch.from_numpy(obs.valid.astype(np.uint8)).to(dev)
            d_more.append((a, d, v, float(obs.distance.max()) if len(obs) else 0.0, odo))
        torch.cuda.synchronize()

        def more_step(i):
            a, d, v, maxd, odo = d_more[i]
            slam.set_scan_device(a.data_ptr(), d.data_ptr(), v.data_ptr(), a.numel(), maxd)
            slam.step_async(odo)
        for i in range(n_more):
            more_step(i)
        slam.sync()
        step0 = slam.stats()["step"]
        barrier()
        e0.record(stream)
        for i in range(n_more, n_more + K):
            more_step(i)
        e1.record(stream)
        slam.sync()
        barrier()
        hist = step_history(slam, step0, K)
        out["aged"] = {"ms": e0.elapsed_time(e1), "scans_before": int(step0), "extent": slam.map_extent(),
                       "particles_integrated_per_step": float(hist[:, 4].mean()), "copy_bytes_per_step": float(hist[:, 5].mean())}
    slam.close()
    return out


def run_cuda(args, wl, rank, world, local):
    import torch
    import torch.distributed as dist
    from slamrs_b200 import nccl_unique_id
    from slamrs_b200 import _lib
    from slamrs_b200.workloads import WORKLOADS

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the CUDA arm has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)

    def fresh_nccl_id():
        if world == 1:
            return None
        buf = torch.zeros(_lib.NCCL_ID_BYTES, dtype=torch.uint8, device=dev)
        if rank == 0:
            buf.copy_(torch.frombuffer(bytearray(nccl_unique_id()), dtype=torch.uint8))
        dist.broadcast(buf, 0)
        return bytes(buf.cpu().numpy().tobytes())

    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    n_total = wl.n_particles * world
    K, W = args.steps, args.warmup
    sim = wl.simulator()
    AGED = 160
    do_aged = not args.no_aged
    scans = [sim.next_scan(wl.speed_left, wl.speed_right) for _ in range(W + 3 * K + ((AGED + K) if do_aged else 0))]

    clocks = ClockSampler(local)
    clocks.start()
    main = measure_cuda(args, wl, rank, world, local, dev, fresh_nccl_id(), scans, args.flags, not args.no_e2e, do_aged)
    clock_info = clocks.stop()
    if not args.no_e2e:
        main["ms_e2e"] = measure_e2e_pipelined(args, wl, rank, world, local, dev, fresh_nccl_id(), scans, args.flags)
    full = None
    # eager / strict are single-GPU diagnostics; the whole-grid-copy leg (the reference's bytes, what the north
    # star's "% of aggregate HBM roofline" describes) also runs sharded
    if world > 1:
        args.no_strict = True
        args.no_eager = True
    if not args.no_full_copy:
        full = measure_cuda(args, wl, rank, world, local, dev, fresh_nccl_id(), scans, _lib.FLAG_FULL_GRID_COPY, False)
    eager = None
    if not args.no_eager:
        eager = measure_cuda(args, wl, rank, world, local, dev, fresh_nccl_id(), scans, _lib.FLAG_EAGER_COPY, False)
    strict = None
    if not args.no_strict:
        strict = measure_cuda(args, wl, rank, world, local, dev, fresh_nccl_id(), scans,
                              _lib.FLAG_UPDATE_ALL_PARTICLES, False)

    def reduce_max(vals):
        t = torch.tensor(vals, dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.cpu().numpy()

    def reduce_sum(vals):
        t = torch.tensor(vals, dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return t.cpu().numpy()

    ph = main["phase_ms"]
    # configs[4] (262,144 x 720 x 2048^2 on 8 GPUs, windowed 512^2 slots, uniform start poses): its own leg
    c5 = None
    if (world == 8 and not args.no_c5) or args.c5_leg:
        wl5 = WORKLOADS["c5"]
        sim5 = wl5.simulator()
        scans5 = [sim5.next_scan(wl5.speed_left, wl5.speed_right) for _ in range(W + K)]
        clocks5 = ClockSampler(local)
        clocks5.start()
        c5 = measure_cuda(args, wl5, rank, world, local, dev, fresh_nccl_id(), scans5, 0, False)
        c5["clocks"] = clocks5.stop()

    # identical state in every mode, or the numbers mean nothing
    hashes = {"default": main["state_sha256"]}
    for name, leg in (("full_grid_copy", full), ("eager_copy", eager), ("strict_order_of_work", strict)):
        if leg:
            hashes[name] = leg["state_sha256"]
    parity_ok = len(set(hashes.values())) == 1

    tmax = reduce_max([main["ms_value"], main.get("ms_e2e", 0.0), strict["ms_value"] if strict else 0.0] +
                      [ph[k] for k in _lib.PHASES] + [full["ms_value"] if full else 0.0, main.get("ms_e2e_window", 0.0),
                                                      eager["ms_value"] if eager else 0.0,
                                                      main["aged"]["ms"] if "aged" in main else 0.0,
                                                      c5["ms_value"] if c5 else 0.0,
                                                      full["phase_ms"]["copy"] if full else 0.0,
                                                      main.get("ms_e2e_sync", 0.0)])
    hist = main["hist"]
    tot = reduce_sum([hist[:, 0].sum(), hist[:, 1].sum(), hist[:, 4].sum(),
                      float(full["hist"][:, 5].sum()) if full else 0.0, float(hist[:, 5].sum()), 8.0 * float(hist[:, 6].sum()),
                      float(c5["hist"][:, 5].sum() + 8.0 * c5["hist"][:, 6].sum()) if c5 else 0.0])
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        if not parity_ok:
            raise SystemExit(3)
        return

    peak, peak_src = measured_peaks()
    pbu = n_total * wl.n_beams
    ms_value, ms_e2e, ms_strict = float(tmax[0]), float(tmax[1]), float(tmax[2])
    grid_bytes = main["grid_bytes"]
    copies, src_reads = hist[:, 0], hist[:, 3]
    # Copy kernels (k_copy_boxed / k_copy), rank 0's own launches: bytes really read + written (device-counted)
    # over the time of the phases they run in (clones made private before the ray update + eager copies / pulls).
    copy_ms = ph["materialize"] + ph["copy"]
    copy_bytes = float(hist[:, 5].sum())
    full_bytes = float(grid_bytes) * (copies.sum() + src_reads.sum())   # what whole-grid copies would move
    copy_roofline = lambda b, ms, kernel: {  # noqa: E731
        "bound": "hbm", "kernel": kernel, "achieved": b / (ms * 1e-3) / 1e9 if ms > 0 else 0.0, "peak": peak, "unit": "GB/s",
        "frac": (b / (ms * 1e-3) / 1e9) / peak if peak and ms > 0 else None, "bytes_per_launch": b / K, "ms_per_launch": ms / K}
    boxed = (int(args.flags) & _lib.FLAG_FULL_GRID_COPY) == 0 and wl.grid % 8 == 0
    deferred = boxed and (int(args.flags) & _lib.FLAG_EAGER_COPY) == 0
    # Ray update (k_ray_update_half): SURVEY.md 8(d)'s unit is the cell-step of the reference's ray iterator,
    # 4 B read + 4 B written each (8 B); the kernel counts the steps of the rays it integrates.
    ray_ms = ph["ray_update"]
    # ... plus the clone copies the same kernel performs (a surviving clone's cells are copied by the CTA that integrates
    # its scan): bytes read + written, counted on the device (history value ray_copy_bytes)
    ray_rmw_bytes = 8.0 * float(hist[:, 6].sum())
    ray_copy_bytes = float(hist[:, 7].sum())
    ray_bytes = ray_rmw_bytes + ray_copy_bytes
    copy_bytes = max(0.0, copy_bytes - ray_copy_bytes)      # what the copy kernels proper moved (NVLink pulls, eager copies)
    st = main["stats"]
    line = {
        "metric": METRIC, "value": pbu * K / (ms_value * 1e-3), "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms_value / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32 geometry, f64 weights, u16x2 hit-counter cells", "data": "synthetic",
        "config": workload_config(wl, world, n_total),
        "clocks": clock_info,
        "gpu_launches": int(main["launches"]),
        "roofline": None,
        "roofline_copy": dict(copy_roofline(copy_bytes, copy_ms, "k_copy_boxed (informed extents, whole 1 KiB tiles)" if boxed
                                            else "k_copy (whole grids)"),
                              traffic=ncu_traffic("copy_traffic.json", copy_bytes / K),
                              grids_copied_per_step=float(copies.mean()), source_reads_per_step=float(src_reads.mean()),
                              bytes_per_grid=int(grid_bytes), whole_grid_bytes_per_launch=full_bytes / K,
                              algorithmic_bytes="bytes the kernel read + wrote per step, counted on the device: informed "
                                                "extent (whole tiles) of every grid written + of every source read"),
        "phases_ms_per_step": {k: float(tmax[3 + i]) / K for i, k in enumerate(_lib.PHASES)},
        "resample": {"grids_copied_per_step_all_gpus": float(tot[0] / K), "grids_pulled_per_step_all_gpus": float(tot[1] / K),
                     "particles_integrated_per_step_all_gpus": float(tot[2] / K),
                     "distinct_sources_last_step_rank0": st["distinct_sources"],
                     "spilled_cells_last_step": st["spilled_cells"], "window_cells": st["window_cells"],
                     "counter_saturated": st["counter_saturated"]},
    }
    ray_roofline = {
        "bound": "hbm", "kernel": "k_ray_update_half (ray walk into a shared-memory half-disc window, then root tiles + window -> own slot "
                                  "with 256-bit accesses: the scan's read-modify-write and the copy of a surviving clone)",
        "achieved": ray_bytes / (ray_ms * 1e-3) / 1e9 if ray_ms > 0 else 0.0, "peak": peak, "unit": "GB/s",
        "frac": (ray_bytes / (ray_ms * 1e-3) / 1e9) / peak if peak and ray_ms > 0 else None,
        "traffic": ncu_traffic("ray_traffic.json", ray_bytes / K), "peak_source": peak_src,
        "bytes_per_launch": ray_bytes / K, "ms_per_launch": ray_ms / K,
        "ray_rmw_bytes_per_launch": ray_rmw_bytes / K, "clone_copy_bytes_per_launch": ray_copy_bytes / K,
        "cell_steps_per_launch": float(hist[:, 6].sum()) / K, "particles_integrated_per_launch": float(hist[:, 4].mean()),
        "algorithmic_bytes": "SURVEY.md 8(d): 8 B (4 read + 4 written) per step of the reference's ray iterator, steps counted "
                             "by the kernel over the rays it integrates, + the bytes of the clone copies the kernel performs "
                             "(2 x informed extent per copied grid, counted on the device). The kernel is bound by instruction "
                             "issue and latency, not by HBM: revisited cells are accumulated in shared memory and every tile "
                             "is read and written once",
        "step_frac": ((ray_bytes + copy_bytes) / (ms_value * 1e-3) / 1e9) / peak if peak else None}
    line["roofline_copy"]["peak_source"] = peak_src
    # the roofline the contract asks for is the dominant kernel's: whichever phase takes more of the step
    if ray_ms >= copy_ms and ray_bytes > 0:
        line["roofline"] = ray_roofline
    else:
        line["roofline"] = dict(line["roofline_copy"], step_frac=(copy_bytes / (ms_value * 1e-3) / 1e9) / peak if peak else None)
        line["roofline_ray_update"] = ray_roofline
    line["deferred_copies"] = bool(deferred)
    line["parity_check"] = {"ok": parity_ok, "state_sha256": hashes,
                            "what": "sha256 over resample indices, argmax, all poses, published pose and published map after the "
                                    "timed steps; every mode must leave the same state (non-zero exit otherwise)"}
    # the whole step against the aggregate roofline of the GPUs it ran on
    line["roofline"]["step_frac_aggregate"] = ((float(tot[4]) + float(tot[5])) / (ms_value * 1e-3) / 1e9) / (peak * world) if peak else None
    if "aged" in main:
        ms_aged = float(tmax[6 + len(_lib.PHASES)])
        line["aged_map"] = {"value": pbu * K / (ms_aged * 1e-3), "unit": UNIT, "ms_per_step": ms_aged / K,
                            "scans_before": main["aged"]["scans_before"], "informed_extent_cells": main["aged"]["extent"],
                            "particles_integrated_per_step_rank0": main["aged"]["particles_integrated_per_step"],
                            "copy_bytes_per_step_rank0": main["aged"]["copy_bytes_per_step"],
                            "note": "the same filter after 160 more scans of the trajectory: informed extents and survivor "
                                    "counts have grown"}
    if c5:
        ms_c5 = float(tmax[7 + len(_lib.PHASES)])
        n5 = WORKLOADS["c5"].n_particles * world
        line["configs4_leg"] = {
            "value": n5 * WORKLOADS["c5"].n_beams * K / (ms_c5 * 1e-3), "unit": UNIT, "ms_per_step": ms_c5 / K,
            "config": workload_config(WORKLOADS["c5"], world, n5), "clocks": c5["clocks"], "state_sha256": c5["state_sha256"],
            "step_frac_aggregate": (float(tot[6]) / (ms_c5 * 1e-3) / 1e9) / (peak * world) if peak else None,
            "phases_ms_per_step_rank0": {k: v / K for k, v in c5["phase_ms"].items()},
            "note": "BASELINE.json configs[4] (one 32,768-particle shard per GPU, 512x512 windowed slots of the 2048^2 grid, "
                    "uniform start poses); complete at 8 GPUs"}
    if "ms_e2e" in main:
        gw, gh = main["grid"]
        line["e2e"] = {"value": pbu * K / (ms_e2e * 1e-3), "unit": UNIT, "ms_per_step": ms_e2e / K,
                       "h2d_bytes_per_step": int(wl.n_beams * (4 + 4 + 1)), "d2h_bytes_per_step": int(12 + 8 * gw * gh),
                       "path": "update(host scan) + estimated_pose() + estimated_likelihood_async() per step, map_wait() before "
                               "the next read-out (node.rs:47-60 with the 8 B/cell map of step t copied to pinned host memory "
                               "while update(t+1) runs; every step's pose and whole map reach the host inside the timed region); "
                               "a filter of its own on the same scans as `value` (W warm-up scans, then the K timed ones)"}
        ms_sync = float(tmax[9 + len(_lib.PHASES)])
        line["e2e_blocking"] = {"value": pbu * K / (ms_sync * 1e-3), "unit": UNIT, "ms_per_step": ms_sync / K,
                                "d2h_bytes_per_step": int(12 + 8 * gw * gh),
                                "path": "update(host scan) + estimated_pose() + estimated_likelihood() per step, each call "
                                        "blocking (node.rs:47-60 as written), on the K scans that follow the `value` leg's"}
        ms_win = float(tmax[4 + len(_lib.PHASES)])
        line["e2e_window_readout"] = {
            "value": pbu * K / (ms_win * 1e-3), "unit": UNIT, "ms_per_step": ms_win / K,
            "d2h_bytes_per_step": int(12 + 16 + main["e2e_window_bytes"]),
            "path": "update(host scan) + estimated_pose() + map_extent() + map_window(f32) per step: the informed "
                    "window of the map instead of 8 B/cell of the whole grid (SURVEY.md 8(f)3)"}
    if full:
        ms_full = float(tmax[3 + len(_lib.PHASES)])
        fh, fph = full["hist"], full["phase_ms"]
        fbytes = float(fh[:, 5].sum())
        line["full_grid_copy"] = {
            "value": pbu * K / (ms_full * 1e-3), "unit": UNIT, "ms_per_step": ms_full / K,
            "note": "SLAMRS_FLAG_FULL_GRID_COPY: every resampling copy moves the whole W*H grid, as Map::clone does "
                    "(particle.rs:97-100); identical results",
            "roofline": dict(copy_roofline(fbytes, float(tmax[8 + len(_lib.PHASES)]) if world > 1 else fph["copy"], "k_copy"),
                             step_frac=(fbytes / (ms_full * 1e-3) / 1e9) / peak if peak else None,
                             step_frac_aggregate=(float(tot[3]) / (ms_full * 1e-3) / 1e9) / (peak * world) if peak else None,
                             note="step_frac_aggregate = bytes all ranks moved per step / step time / (n_gpus x measured HBM "
                                  "peak): the north star's '% of aggregate HBM roofline per SLAM step'"),
            "phases_ms_per_step": {k: v / K for k, v in fph.items()}}
    if eager:
        ms_eager = float(tmax[5 + len(_lib.PHASES)])
        eh, eph = eager["hist"], eager["phase_ms"]
        ebytes = float(eh[:, 5].sum())
        line["eager_copy"] = {
            "value": pbu * K / (ms_eager * 1e-3), "unit": UNIT, "ms_per_step": ms_eager / K,
            "note": "SLAMRS_FLAG_EAGER_COPY: every clone is copied when resampling creates it (informed extent only), as "
                    "value.clone() does (particle.rs:97-100); the default copies a clone when it is first written",
            "roofline": copy_roofline(ebytes, eph["materialize"] + eph["copy"], "k_copy_boxed"),
            "grids_copied_per_step": float(eh[:, 0].mean()),
            "phases_ms_per_step": {k: v / K for k, v in eph.items()}}
    if strict:
        line["strict_order_of_work"] = {
            "value": pbu * K / (ms_strict * 1e-3), "unit": UNIT, "ms_per_step": ms_strict / K,
            "note": "SLAMRS_FLAG_UPDATE_ALL_PARTICLES: the scan is integrated into every particle's grid before "
                    "resampling, as the reference orders the work; results are identical to the default, which "
                    "integrates only the grids that survive the step's resampling",
            "phases_ms_per_step": {k: v / K for k, v in strict["phase_ms"].items()}}
    if world == 1 and not args.no_cpu_baseline:
        from oracle import oracle as O
        cores = os.cpu_count() or 1
        n_cpu = args.cpu_particles or max(cores * 8, 64)
        res = time_oracle(O, wl, n_cpu, steps=6, warmup=2, threads=cores)
        res1 = time_oracle(O, wl, max(16, n_cpu // 8), steps=4, warmup=1, threads=1)
        resd = time_oracle(O, wl, max(16, n_cpu // 8), steps=3, warmup=1, threads=1, dead_likelihood=True)
        line["cpu_baseline"] = {"value": res["value"], "unit": UNIT, "cores": cores, "kind": "port",
                                "sample": res["sample"], "single_thread_value": res1["value"],
                                "single_thread_sample": res1["sample"],
                                "single_thread_with_dead_likelihood_value": resd["value"],
                                "single_thread_with_dead_likelihood_sample": resd["sample"],
                                "note": "C restatement of the Rust reference (no Rust toolchain in the image). The reference "
                                        "itself is single-threaded (particle.rs:32-35) and, unless rustc elides it, also runs "
                                        "the dead Map::likelihood() transform per particle (slam.rs:58): the two single_thread "
                                        "values bracket it. `value` (all host threads, no dead transform) is the generous "
                                        "figure and the one the --impl reference arm reports, i.e. what the driver's "
                                        "vs_reference ratio divides by"}
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, main["outputs"])
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    if not parity_ok:
        raise SystemExit("bench.py: the comparison modes left different filter states: " + json.dumps(hashes))


def ncu_traffic(name, bytes_per_launch):
    """DRAM bytes per launch of a kernel from the committed ncu --set full capture (profiles/<name> holds
    dram__bytes_read + dram__bytes_write per algorithmic byte of that capture)."""
    path = os.path.join(ROOT, "profiles", name)
    if not os.path.exists(path):
        return None
    with open(path) as f:
        ratio = json.load(f)["dram_bytes_per_algorithmic_byte"]
    return ratio * bytes_per_launch


def cfg_cells(slam):
    return slam.grid_w * slam.grid_h


def main():
    args = parse_args()
    rank, world, local = dist_env()
    if world == 1 and args.gpus > 1 and args.impl == "cuda":
        raise SystemExit("bench.py: --gpus N>1 must be launched with torch.distributed.run (one rank per GPU)")
    from slamrs_b200.workloads import WORKLOADS
    wl = WORKLOADS[args.workload]
    if args.particles:
        import dataclasses
        wl = dataclasses.replace(wl, n_particles=args.particles)
    if args.impl == "reference":
        run_reference(args, wl, rank, world)
    else:
        run_cuda(args, wl, rank, world, local)


if __name__ == "__main__":
    main()
