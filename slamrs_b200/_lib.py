"""ctypes binding of include/slamrs_gpu.h. There is no CPU fallback: if the CUDA library is
missing it is built with nvcc, and if that fails the import error is raised to the caller."""
from __future__ import annotations

import ctypes as C
import os

from . import build as _build

NCCL_ID_BYTES = 128
ABI_VERSION = 1

OK = 0
E_INVALID_ARG, E_CUDA, E_NCCL, E_OOM, E_NO_DEVICE, E_STAGING, E_NOT_LOCAL, E_INTERNAL = -1, -2, -3, -4, -5, -6, -7, -8
E_WINDOW = -9
RNG_SHARED_STREAM, RNG_CALLER = 0, 1
FLAG_GENERIC_RAY_KERNEL = 1
FLAG_UPDATE_ALL_PARTICLES = 2
FLAG_FULL_GRID_COPY = 4
FLAG_NCCL_EXCHANGE = 8
FLAG_EAGER_COPY = 16
FLAG_SERIAL_STEPS = 32
HISTORY_VALUES = 8

EXPORTS = [
    "slamrs_gpu_grid_cells", "slamrs_gpu_nccl_unique_id", "slamrs_gpu_create", "slamrs_gpu_destroy",
    "slamrs_gpu_update", "slamrs_gpu_upload_scan", "slamrs_gpu_step_async", "slamrs_gpu_sync",
    "slamrs_gpu_pose", "slamrs_gpu_map_probability", "slamrs_gpu_last_error", "slamrs_gpu_get_stats",
    "slamrs_gpu_stream", "slamrs_gpu_launch_count", "slamrs_gpu_get_poses", "slamrs_gpu_set_poses",
    "slamrs_gpu_get_weights", "slamrs_gpu_get_resample_indices", "slamrs_gpu_get_max_particle",
    "slamrs_gpu_get_cells", "slamrs_gpu_set_cells", "slamrs_gpu_get_log_odds",
    "slamrs_gpu_debug_raycast", "slamrs_gpu_debug_sincos", "slamrs_gpu_debug_stream",
    "slamrs_gpu_set_scan_device", "slamrs_gpu_set_profiling", "slamrs_gpu_get_phase_ms",
    "slamrs_gpu_get_step_history", "slamrs_gpu_map_extent", "slamrs_gpu_map_window",
    "slamrs_gpu_effective_particles", "slamrs_gpu_sim_scan", "slamrs_gpu_get_scan", "slamrs_gpu_get_slots",
    "slamrs_gpu_get_extents", "slamrs_gpu_debug_resample", "slamrs_gpu_debug_resample_adaptive", "slamrs_gpu_init_uniform",
    "slamrs_gpu_map_probability_async", "slamrs_gpu_map_wait",
    "slamrs_gpu_create_localizer", "slamrs_gpu_get_sensor_terms",
    "slamrs_gpu_set_scan_match", "slamrs_gpu_get_scan_match_stats",
    "slamrs_gpu_set_recovery", "slamrs_gpu_get_recovery_state",
    "slamrs_gpu_set_kld", "slamrs_gpu_get_kld_state", "slamrs_gpu_get_population",
    "slamrs_gpu_pose_clusters",
]
MAP_F64, MAP_F32, MAP_U8 = 0, 1, 2
SENSOR_BEAM_ENDPOINT, SENSOR_LIKELIHOOD_FIELD = 0, 1
PHASES = ["motion_likelihood", "all_gather", "resample", "materialize", "ray_update", "pull", "copy"]


class Config(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32), ("abi_version", C.c_uint32),
        ("pos_x", C.c_float), ("pos_y", C.c_float), ("resolution", C.c_float),
        ("grid_w", C.c_uint32), ("grid_h", C.c_uint32),
        ("n_particles", C.c_uint64), ("seed", C.c_uint64),
        ("rng_mode", C.c_uint32), ("device", C.c_int32),
        ("rank", C.c_uint32), ("world_size", C.c_uint32),
        ("spare_slots", C.c_uint32), ("flags", C.c_uint32),
        ("slot_cells", C.c_uint32), ("resample_threshold", C.c_float),
        ("nccl_id", C.c_uint8 * NCCL_ID_BYTES),
    ]


class SensorModel(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("kind", C.c_uint32), ("sigma", C.c_float), ("z_rand", C.c_float),
                ("occupied_above", C.c_float)]


class ScanMatch(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("radius", C.c_uint32), ("step_xy", C.c_float), ("step_theta", C.c_float),
                ("levels", C.c_uint32), ("max_moves", C.c_uint32)]


class Recovery(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("pad", C.c_uint32), ("alpha_slow", C.c_double), ("alpha_fast", C.c_double)]


class Kld(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("n_min", C.c_uint32), ("n_max", C.c_uint32), ("pad", C.c_uint32),
                ("err", C.c_double), ("z", C.c_double), ("bin_cells", C.c_uint32), ("theta_bins", C.c_uint32)]


class Clustering(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("bin_cells", C.c_uint32), ("theta_bins", C.c_uint32),
                ("max_clusters", C.c_uint32)]


class PoseCluster(C.Structure):
    _fields_ = [("count", C.c_uint64), ("label", C.c_uint64), ("weight", C.c_double), ("mean", C.c_double * 3),
                ("cov_xx", C.c_double), ("cov_xy", C.c_double), ("cov_yy", C.c_double), ("var_theta", C.c_double)]


class PoseStats(C.Structure):
    _fields_ = [("n_poses", C.c_uint64), ("n_excluded", C.c_uint64), ("n_bins", C.c_uint64), ("n_clusters", C.c_uint64),
                ("overall", PoseCluster)]


class Stats(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in (
        "step", "grids_copied", "grids_pulled", "distinct_sources", "resample_clamped",
        "counter_saturated", "spilled_cells", "window_cells", "bytes_per_grid", "particles_integrated",
        "copy_bytes", "window_overflow", "resample_exact_fallback", "resample_fold_rounds", "resampled")]


class SlamrsGpuError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"slamrs_gpu error {code}: {msg}")
        self.code = code


_lib = None


def lib_path() -> str:
    return _build.LIB


def load():
    """Load (building first if needed) libslamrs_gpu.so and declare every prototype."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.build() if _build.needs_build() else _build.LIB
    path = os.environ.get("SLAMRS_GPU_LIB", path)   # tuning variants built by `python slamrs_b200/build.py -D... --out=...`
    L = C.CDLL(path, mode=C.RTLD_GLOBAL)
    vp, u32, u64, f, i = C.c_void_p, C.c_uint32, C.c_uint64, C.c_float, C.c_int
    L.slamrs_gpu_grid_cells.restype = i; L.slamrs_gpu_grid_cells.argtypes = [f, f, C.POINTER(u32)]
    L.slamrs_gpu_nccl_unique_id.restype = i; L.slamrs_gpu_nccl_unique_id.argtypes = [vp]
    L.slamrs_gpu_create.restype = i; L.slamrs_gpu_create.argtypes = [C.POINTER(Config), C.POINTER(vp)]
    L.slamrs_gpu_destroy.restype = None; L.slamrs_gpu_destroy.argtypes = [vp]
    L.slamrs_gpu_update.restype = i
    L.slamrs_gpu_update.argtypes = [vp, vp, vp, vp, u32, f, f, f, vp, vp]
    L.slamrs_gpu_upload_scan.restype = i; L.slamrs_gpu_upload_scan.argtypes = [vp, vp, vp, vp, u32]
    L.slamrs_gpu_step_async.restype = i; L.slamrs_gpu_step_async.argtypes = [vp, f, f, f, vp, vp]
    L.slamrs_gpu_sync.restype = i; L.slamrs_gpu_sync.argtypes = [vp]
    L.slamrs_gpu_pose.restype = i; L.slamrs_gpu_pose.argtypes = [vp, vp]
    L.slamrs_gpu_map_probability.restype = i; L.slamrs_gpu_map_probability.argtypes = [vp, vp]
    L.slamrs_gpu_map_probability_async.restype = i; L.slamrs_gpu_map_probability_async.argtypes = [vp, vp]
    L.slamrs_gpu_map_wait.restype = i; L.slamrs_gpu_map_wait.argtypes = [vp]
    L.slamrs_gpu_last_error.restype = C.c_char_p; L.slamrs_gpu_last_error.argtypes = [vp]
    L.slamrs_gpu_get_stats.restype = i; L.slamrs_gpu_get_stats.argtypes = [vp, C.POINTER(Stats)]
    L.slamrs_gpu_stream.restype = vp; L.slamrs_gpu_stream.argtypes = [vp]
    L.slamrs_gpu_launch_count.restype = u64; L.slamrs_gpu_launch_count.argtypes = [vp]
    L.slamrs_gpu_get_poses.restype = i; L.slamrs_gpu_get_poses.argtypes = [vp, vp]
    L.slamrs_gpu_set_poses.restype = i; L.slamrs_gpu_set_poses.argtypes = [vp, vp]
    L.slamrs_gpu_get_weights.restype = i; L.slamrs_gpu_get_weights.argtypes = [vp, vp, vp]
    L.slamrs_gpu_get_resample_indices.restype = i; L.slamrs_gpu_get_resample_indices.argtypes = [vp, vp]
    L.slamrs_gpu_get_max_particle.restype = i; L.slamrs_gpu_get_max_particle.argtypes = [vp, C.POINTER(u64)]
    L.slamrs_gpu_get_cells.restype = i; L.slamrs_gpu_get_cells.argtypes = [vp, u64, vp]
    L.slamrs_gpu_set_cells.restype = i; L.slamrs_gpu_set_cells.argtypes = [vp, u64, vp]
    L.slamrs_gpu_get_log_odds.restype = i; L.slamrs_gpu_get_log_odds.argtypes = [vp, u64, vp]
    L.slamrs_gpu_debug_raycast.restype = i
    L.slamrs_gpu_debug_raycast.argtypes = [i, vp, vp, vp, vp, u32, u32, u32, u32, vp, u32, vp]
    L.slamrs_gpu_debug_sincos.restype = i; L.slamrs_gpu_debug_sincos.argtypes = [i, vp, u32, vp, vp]
    L.slamrs_gpu_debug_stream.restype = i; L.slamrs_gpu_debug_stream.argtypes = [i, u64, u64, u64, u64, vp, vp]
    L.slamrs_gpu_set_scan_device.restype = i; L.slamrs_gpu_set_scan_device.argtypes = [vp, vp, vp, vp, u32, f]
    L.slamrs_gpu_set_profiling.restype = i; L.slamrs_gpu_set_profiling.argtypes = [vp, i]
    L.slamrs_gpu_get_phase_ms.restype = i; L.slamrs_gpu_get_phase_ms.argtypes = [vp, vp, C.POINTER(u64)]
    L.slamrs_gpu_get_step_history.restype = i; L.slamrs_gpu_get_step_history.argtypes = [vp, u64, u32, vp]
    L.slamrs_gpu_map_extent.restype = i; L.slamrs_gpu_map_extent.argtypes = [vp, vp]
    L.slamrs_gpu_map_window.restype = i
    L.slamrs_gpu_map_window.argtypes = [vp, u32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, vp]
    L.slamrs_gpu_effective_particles.restype = i
    L.slamrs_gpu_effective_particles.argtypes = [vp, C.POINTER(C.c_double)]
    L.slamrs_gpu_sim_scan.restype = i; L.slamrs_gpu_sim_scan.argtypes = [vp, vp, u32, vp, u32, f, C.POINTER(u32)]
    L.slamrs_gpu_get_scan.restype = i; L.slamrs_gpu_get_scan.argtypes = [vp, vp, vp, vp, u32, C.POINTER(u32)]
    L.slamrs_gpu_get_slots.restype = i; L.slamrs_gpu_get_slots.argtypes = [vp, vp, vp, C.POINTER(u32)]
    L.slamrs_gpu_get_extents.restype = i; L.slamrs_gpu_get_extents.argtypes = [vp, u64, vp, vp, C.POINTER(u32)]
    L.slamrs_gpu_init_uniform.restype = i; L.slamrs_gpu_init_uniform.argtypes = [vp, vp]
    L.slamrs_gpu_create_localizer.restype = i
    L.slamrs_gpu_create_localizer.argtypes = [C.POINTER(Config), C.POINTER(SensorModel), vp, C.POINTER(vp)]
    L.slamrs_gpu_get_sensor_terms.restype = i; L.slamrs_gpu_get_sensor_terms.argtypes = [vp, vp]
    L.slamrs_gpu_set_scan_match.restype = i; L.slamrs_gpu_set_scan_match.argtypes = [vp, C.POINTER(ScanMatch)]
    L.slamrs_gpu_get_scan_match_stats.restype = i; L.slamrs_gpu_get_scan_match_stats.argtypes = [vp, vp]
    L.slamrs_gpu_set_recovery.restype = i; L.slamrs_gpu_set_recovery.argtypes = [vp, C.POINTER(Recovery)]
    L.slamrs_gpu_get_recovery_state.restype = i; L.slamrs_gpu_get_recovery_state.argtypes = [vp, vp, C.POINTER(u64)]
    L.slamrs_gpu_set_kld.restype = i; L.slamrs_gpu_set_kld.argtypes = [vp, C.POINTER(Kld)]
    L.slamrs_gpu_get_kld_state.restype = i; L.slamrs_gpu_get_kld_state.argtypes = [vp, vp]
    L.slamrs_gpu_get_population.restype = i; L.slamrs_gpu_get_population.argtypes = [vp, C.POINTER(u64)]
    L.slamrs_gpu_pose_clusters.restype = i
    L.slamrs_gpu_pose_clusters.argtypes = [vp, C.POINTER(Clustering), C.POINTER(PoseStats), vp]
    L.slamrs_gpu_debug_resample.restype = i
    L.slamrs_gpu_debug_resample.argtypes = [i, vp, u32, C.c_double, vp, C.POINTER(u64), vp, vp, vp, vp]
    L.slamrs_gpu_debug_resample_adaptive.restype = i
    L.slamrs_gpu_debug_resample_adaptive.argtypes = [i, vp, u32, C.c_double, C.c_double, vp, C.POINTER(u64), vp, vp, vp,
                                                     vp, C.POINTER(C.c_double), C.POINTER(u64), vp]
    _lib = L
    return L


def check(rc: int, handle=None):
    if rc != OK:
        msg = load().slamrs_gpu_last_error(handle)
        raise SlamrsGpuError(rc, msg.decode() if msg else "")
