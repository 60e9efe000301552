"""CPU-side checks: the C-ABI library loads and exports every symbol include/slamrs_gpu.h
declares, fails loudly without a GPU (no CPU fallback), and the host-side logic (grid sizing,
scan generator, workloads) behaves like the reference."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import slamrs_b200
from slamrs_b200 import _lib
from slamrs_b200.simulator import Simulator, reference_scene, scan
from slamrs_b200.workloads import WORKLOADS

from common import gpu_present

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "slamrs_gpu.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(slamrs_gpu_\w+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    L = _lib.load()
    declared = _declared_symbols()
    assert len(declared) >= 25
    for name in declared:
        assert hasattr(L, name), f"{name} declared in include/slamrs_gpu.h but not exported"
    assert sorted(_lib.EXPORTS) == declared, "python binding list out of sync with the header"


def test_config_struct_matches_header_layout():
    # uint32 x2, float x3, uint32 x2, (pad) uint64 x2, uint32, int32, uint32 x4, 128 bytes
    assert C.sizeof(_lib.Config) == 208
    assert _lib.Config.n_particles.offset == 32 and _lib.Config.nccl_id.offset == 80
    assert C.sizeof(_lib.Stats) == 120


def test_product_does_not_touch_the_oracle():
    """The shipped package and library must never import, link or call oracle/."""
    pkg = os.path.join(ROOT, "slamrs_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp", ".hpp")):
                src = open(os.path.join(dirpath, f)).read()
                assert "liboracle" not in src and "slam_oracle" not in src, f
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), f


@pytest.mark.skipif(gpu_present(), reason="GPU present")
def test_no_gpu_means_loud_error_not_fallback():
    with pytest.raises(_lib.SlamrsGpuError) as e:
        slamrs_b200.GridMapSlam(slamrs_b200.GridMapSlamConfig(n_particles=4))
    assert e.value.code == _lib.E_NO_DEVICE
    assert "no CPU fallback" in str(e.value)


def test_argument_validation_without_gpu():
    L = _lib.load()
    h = C.c_void_p()
    assert L.slamrs_gpu_create(None, C.byref(h)) == _lib.E_INVALID_ARG
    cfg = _lib.Config()
    cfg.struct_size = 12                              # wrong size -> ABI mismatch
    assert L.slamrs_gpu_create(C.byref(cfg), C.byref(h)) == _lib.E_INVALID_ARG
    cfg.struct_size = C.sizeof(_lib.Config); cfg.abi_version = _lib.ABI_VERSION
    cfg.n_particles = 0; cfg.grid_w = cfg.grid_h = 8; cfg.resolution = 0.1; cfg.world_size = 1
    assert L.slamrs_gpu_create(C.byref(cfg), C.byref(h)) == _lib.E_INVALID_ARG   # particle.rs:16 assert
    assert b"at least one particle" in L.slamrs_gpu_last_error(None)
    cfg.n_particles = 4; cfg.grid_h = 4
    assert L.slamrs_gpu_create(C.byref(cfg), C.byref(h)) == _lib.E_INVALID_ARG   # non-square
    cfg.grid_h = 8; cfg.world_size = 3
    assert L.slamrs_gpu_create(C.byref(cfg), C.byref(h)) == _lib.E_INVALID_ARG   # 4 % 3 != 0
    assert L.slamrs_gpu_update(None, None, None, None, 0, 0, 0, 0, None, None) == _lib.E_INVALID_ARG
    L.slamrs_gpu_destroy(None)                                                    # safe on NULL


def test_grid_sizing_matches_map_new(oracle):
    # map.rs:28-31: ceil(width / resolution) in f32
    for extent, res in [(4.0, 0.02), (8.0, 0.02), (25.6, 0.05), (51.2, 0.05), (102.4, 0.05), (4.02, 0.02), (1.0, 0.3)]:
        assert slamrs_b200.grid_cells(extent, res) == oracle.grid_cells(extent, res)
    assert [slamrs_b200.grid_cells(w, r) for w, r in [(4.0, 0.02), (25.6, 0.05), (51.2, 0.05)]] == [200, 512, 1024]


def test_scan_generator_matches_oracle_simulator(oracle):
    for scale, rng_range, pose in [(1.0, 1.0, (0, 0, 0)), (5.0, 6.0, (0.3, -0.2, 0.7)), (10.0, 6.0, (1.0, 2.0, -2.0))]:
        obs = scan(reference_scene(scale), pose, 360, rng_range)
        a, d, v = oracle.sim_scan(reference_scene(scale), pose, 360, rng_range)
        assert len(obs) == len(a)
        assert np.array_equal(obs.valid, v.astype(bool))
        assert np.allclose(obs.angle, a, atol=1e-6) and np.allclose(obs.distance, d, atol=1e-5)
    assert int(scan(reference_scene(1.0), (0, 0, 0), 360, 1.0).valid.sum()) == 222   # slamrs/out.log:4


def test_simulator_odometry_and_workloads():
    w = WORKLOADS["c1"]
    sim = w.simulator()
    obs, odo = sim.next_scan(w.speed_left, w.speed_right)
    assert len(obs) == 360
    # 30 ticks of f32 1/30 s accumulate to just over 1.0, which trips `timer > update_period` (sim.rs:110-111)
    assert odo.distance_left == pytest.approx(0.08, rel=1e-5)
    assert odo.distance_right == pytest.approx(0.10, rel=1e-5)
    for key, grid in [("c1", 200), ("c2", 512), ("c3", 1024)]:
        cfg = WORKLOADS[key].slam_config()
        assert slamrs_b200.grid_cells(cfg.width, cfg.resolution) == grid
        assert slamrs_b200.grid_cells(cfg.height, cfg.resolution) == grid


def test_ray_walk_loop_compiled_to_the_tight_form():
    """The tested free-run loop of the walk in both packed kernels must stay one predicated block without the
    in-loop rebuild of the row table's shared address (tools/sass_hot_loop.py; the slow form cost 15 % of the
    kernel on B200)."""
    import shutil
    import sys
    if shutil.which("cuobjdump") is None:
        pytest.skip("cuobjdump not installed")
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    from sass_hot_loop import hot_loop
    for kernel in ("k_ray_update_packed", "k_ray_update_half"):
        r = hot_loop(os.path.join(ROOT, "slamrs_b200", "libslamrs_gpu.so"), kernel)
        assert not r["s2ur"] and not r["local_memory"], (kernel, r["body"])
        assert r["instructions"] <= 27, (kernel, r["instructions"])


def test_bindings_agree_with_the_header_on_flags_phases_and_history():
    text = open(os.path.join(ROOT, "include", "slamrs_gpu.h")).read()
    flags = dict(re.findall(r"SLAMRS_FLAG_(\w+)\s*=\s*(\d+)", text))
    assert {k: int(v) for k, v in flags.items()} == {
        "GENERIC_RAY_KERNEL": _lib.FLAG_GENERIC_RAY_KERNEL, "UPDATE_ALL_PARTICLES": _lib.FLAG_UPDATE_ALL_PARTICLES,
        "FULL_GRID_COPY": _lib.FLAG_FULL_GRID_COPY, "NCCL_EXCHANGE": _lib.FLAG_NCCL_EXCHANGE,
        "EAGER_COPY": _lib.FLAG_EAGER_COPY}
    phases = re.findall(r"SLAMRS_PHASE_(\w+)\s*=\s*(\d+)", text)
    names = [n.lower() for n, v in sorted(phases, key=lambda nv: int(nv[1])) if n != "COUNT"]
    assert names == _lib.PHASES
    assert int(re.search(r"#define SLAMRS_HISTORY_VALUES (\d+)", text).group(1)) == _lib.HISTORY_VALUES
    rust = open(os.path.join(ROOT, "rust", "slam-gpu-sys", "src", "lib.rs")).read()
    assert int(re.search(r"SLAMRS_HISTORY_VALUES: usize = (\d+)", rust).group(1)) == _lib.HISTORY_VALUES
    for name, value in flags.items():
        assert re.search(rf"SLAMRS_FLAG_{name}: u32 = {value};", rust), name
