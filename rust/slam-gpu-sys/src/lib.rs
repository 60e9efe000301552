//! Raw bindings, one item per declaration of `include/slamrs_gpu.h` (ABI version 1).
#![allow(non_camel_case_types)]
use core::ffi::{c_char, c_int, c_void};

pub const SLAMRS_GPU_ABI_VERSION: u32 = 1;
pub const SLAMRS_NCCL_ID_BYTES: usize = 128;

pub const SLAMRS_OK: c_int = 0;
pub const SLAMRS_E_INVALID_ARG: c_int = -1;
pub const SLAMRS_E_CUDA: c_int = -2;
pub const SLAMRS_E_NCCL: c_int = -3;
pub const SLAMRS_E_OUT_OF_MEMORY: c_int = -4;
pub const SLAMRS_E_NO_DEVICE: c_int = -5;
pub const SLAMRS_E_STAGING: c_int = -6;
pub const SLAMRS_E_NOT_LOCAL: c_int = -7;
pub const SLAMRS_E_INTERNAL: c_int = -8;
pub const SLAMRS_E_WINDOW: c_int = -9;

pub const SLAMRS_RNG_SHARED_STREAM: u32 = 0;
pub const SLAMRS_RNG_CALLER: u32 = 1;

pub const SLAMRS_FLAG_GENERIC_RAY_KERNEL: u32 = 1;
pub const SLAMRS_FLAG_UPDATE_ALL_PARTICLES: u32 = 2;
pub const SLAMRS_FLAG_FULL_GRID_COPY: u32 = 4;
pub const SLAMRS_FLAG_NCCL_EXCHANGE: u32 = 8;
pub const SLAMRS_FLAG_EAGER_COPY: u32 = 16;

pub const SLAMRS_MAP_F64: u32 = 0;
pub const SLAMRS_MAP_F32: u32 = 1;
pub const SLAMRS_MAP_U8: u32 = 2;
pub const SLAMRS_HISTORY_VALUES: usize = 8;

pub const SLAMRS_SENSOR_BEAM_ENDPOINT: u32 = 0;
pub const SLAMRS_SENSOR_LIKELIHOOD_FIELD: u32 = 1;

#[repr(C)]
pub struct slamrs_gpu_handle {
    _private: [u8; 0],
}

#[repr(C)]
#[derive(Clone, Copy)]
pub struct slamrs_gpu_config {
    pub struct_size: u32,
    pub abi_version: u32,
    pub pos_x: f32,
    pub pos_y: f32,
    pub resolution: f32,
    pub grid_w: u32,
    pub grid_h: u32,
    pub n_particles: u64,
    pub seed: u64,
    pub rng_mode: u32,
    pub device: i32,
    pub rank: u32,
    pub world_size: u32,
    pub spare_slots: u32,
    pub flags: u32,
    pub slot_cells: u32,
    pub resample_threshold: f32,
    pub nccl_id: [u8; SLAMRS_NCCL_ID_BYTES],
}

#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct slamrs_gpu_stats {
    pub step: u64,
    pub grids_copied: u64,
    pub grids_pulled: u64,
    pub distinct_sources: u64,
    pub resample_clamped: u64,
    pub counter_saturated: u64,
    pub spilled_cells: u64,
    pub window_cells: u64,
    pub bytes_per_grid: u64,
    pub particles_integrated: u64,
    pub copy_bytes: u64,
    pub window_overflow: u64,
    pub resample_exact_fallback: u64,
    pub resample_fold_rounds: u64,
    pub resampled: u64,
}

#[repr(C)]
#[derive(Clone, Copy)]
pub struct slamrs_gpu_sensor_model {
    pub struct_size: u32,
    pub kind: u32,
    pub sigma: f32,
    pub z_rand: f32,
    pub occupied_above: f32,
}

#[repr(C)]
#[derive(Clone, Copy)]
pub struct slamrs_gpu_scan_match {
    pub struct_size: u32,
    pub radius: u32,
    pub step_xy: f32,
    pub step_theta: f32,
    pub levels: u32,
    pub max_moves: u32,
}

extern "C" {
    pub fn slamrs_gpu_grid_cells(extent: f32, resolution: f32, out_cells: *mut u32) -> c_int;
    pub fn slamrs_gpu_nccl_unique_id(out: *mut u8) -> c_int;
    pub fn slamrs_gpu_create(cfg: *const slamrs_gpu_config, out: *mut *mut slamrs_gpu_handle) -> c_int;
    pub fn slamrs_gpu_destroy(h: *mut slamrs_gpu_handle);
    pub fn slamrs_gpu_update(
        h: *mut slamrs_gpu_handle,
        angle: *const f32,
        dist: *const f32,
        valid: *const u8,
        n_beams: u32,
        dist_left: f32,
        dist_right: f32,
        wheel_dist: f32,
        z_draws: *const f64,
        resample_u: *const f64,
    ) -> c_int;
    pub fn slamrs_gpu_upload_scan(h: *mut slamrs_gpu_handle, angle: *const f32, dist: *const f32, valid: *const u8, n_beams: u32) -> c_int;
    pub fn slamrs_gpu_step_async(h: *mut slamrs_gpu_handle, dist_left: f32, dist_right: f32, wheel_dist: f32, z_draws: *const f64, resample_u: *const f64) -> c_int;
    pub fn slamrs_gpu_sync(h: *mut slamrs_gpu_handle) -> c_int;
    pub fn slamrs_gpu_set_scan_device(h: *mut slamrs_gpu_handle, angle: *const f32, dist: *const f32, valid: *const u8, n_beams: u32, max_dist: f32) -> c_int;
    pub fn slamrs_gpu_pose(h: *mut slamrs_gpu_handle, out_xyt: *mut f32) -> c_int;
    pub fn slamrs_gpu_map_probability(h: *mut slamrs_gpu_handle, out_cells: *mut f64) -> c_int;
    pub fn slamrs_gpu_map_probability_async(h: *mut slamrs_gpu_handle, out_cells: *mut f64) -> c_int;
    pub fn slamrs_gpu_map_wait(h: *mut slamrs_gpu_handle) -> c_int;
    pub fn slamrs_gpu_map_extent(h: *mut slamrs_gpu_handle, out_x0y0x1y1: *mut i32) -> c_int;
    pub fn slamrs_gpu_map_window(h: *mut slamrs_gpu_handle, format: u32, x0: i32, y0: i32, x1: i32, y1: i32, out: *mut c_void) -> c_int;
    pub fn slamrs_gpu_effective_particles(h: *mut slamrs_gpu_handle, out: *mut f64) -> c_int;
    pub fn slamrs_gpu_init_uniform(h: *mut slamrs_gpu_handle, box_x0y0x1y1: *const f32) -> c_int;
    pub fn slamrs_gpu_sim_scan(h: *mut slamrs_gpu_handle, segments_xyxy: *const f32, n_segments: u32, pose_xyt: *const f32, n_beams: u32, scanner_range: f32, out_n: *mut u32) -> c_int;
    pub fn slamrs_gpu_get_scan(h: *mut slamrs_gpu_handle, out_angle: *mut f32, out_dist: *mut f32, out_valid: *mut u8, cap: u32, out_n: *mut u32) -> c_int;
    pub fn slamrs_gpu_last_error(h: *const slamrs_gpu_handle) -> *const c_char;
    pub fn slamrs_gpu_get_stats(h: *mut slamrs_gpu_handle, out: *mut slamrs_gpu_stats) -> c_int;
    pub fn slamrs_gpu_stream(h: *mut slamrs_gpu_handle) -> *mut c_void;
    pub fn slamrs_gpu_launch_count(h: *const slamrs_gpu_handle) -> u64;
    pub fn slamrs_gpu_set_profiling(h: *mut slamrs_gpu_handle, enabled: c_int) -> c_int;
    pub fn slamrs_gpu_get_phase_ms(h: *mut slamrs_gpu_handle, out_ms: *mut f64, out_steps: *mut u64) -> c_int;
    pub fn slamrs_gpu_get_step_history(h: *mut slamrs_gpu_handle, first_step: u64, count: u32, out_values: *mut u64) -> c_int;
    pub fn slamrs_gpu_get_poses(h: *mut slamrs_gpu_handle, out_xyt: *mut f32) -> c_int;
    pub fn slamrs_gpu_set_poses(h: *mut slamrs_gpu_handle, xyt: *const f32) -> c_int;
    pub fn slamrs_gpu_get_slots(h: *mut slamrs_gpu_handle, out_slot_of: *mut i32, out_spare: *mut i32, out_n_spare: *mut u32) -> c_int;
    pub fn slamrs_gpu_get_weights(h: *mut slamrs_gpu_handle, out_norm: *mut f64, out_raw: *mut f64) -> c_int;
    pub fn slamrs_gpu_get_resample_indices(h: *mut slamrs_gpu_handle, out_idx: *mut u32) -> c_int;
    pub fn slamrs_gpu_get_max_particle(h: *mut slamrs_gpu_handle, out: *mut u64) -> c_int;
    pub fn slamrs_gpu_get_cells(h: *mut slamrs_gpu_handle, particle: u64, out_cells: *mut u32) -> c_int;
    pub fn slamrs_gpu_set_cells(h: *mut slamrs_gpu_handle, particle: u64, cells: *const u32) -> c_int;
    pub fn slamrs_gpu_get_extents(h: *mut slamrs_gpu_handle, particle: u64, out_box_shift: *mut i32, out_bands: *mut u32, out_n_bands: *mut u32) -> c_int;
    pub fn slamrs_gpu_create_localizer(cfg: *const slamrs_gpu_config, model: *const slamrs_gpu_sensor_model, map_probability: *const f64, out: *mut *mut slamrs_gpu_handle) -> c_int;
    pub fn slamrs_gpu_get_sensor_terms(h: *mut slamrs_gpu_handle, out_cells: *mut f64) -> c_int;
    pub fn slamrs_gpu_get_log_odds(h: *mut slamrs_gpu_handle, particle: u64, out_cells: *mut f64) -> c_int;
    pub fn slamrs_gpu_set_scan_match(h: *mut slamrs_gpu_handle, m: *const slamrs_gpu_scan_match) -> c_int;
    pub fn slamrs_gpu_get_scan_match_stats(h: *mut slamrs_gpu_handle, out: *mut u64) -> c_int;
}
