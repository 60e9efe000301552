/* slamrs_gpu.h -- C ABI of the B200-native grid particle-filter SLAM step.
 *
 * This is the drop-in boundary behind slamrs' unchanged `GridMapSlamNode`
 * (slamrs/slam/src/grid/node.rs:35-60). The reference has no FFI; the seam is the inherent API
 * of `struct GridMapSlam` (slamrs/slam/src/grid/slam.rs:13-97). Each entry point below names the
 * Rust item it replaces. INTEGRATION.md shows the Rust `-sys` binding a maintainer would add.
 *
 * Conventions
 *   - every function returns an int status: 0 = SLAMRS_OK, negative = error (see enum);
 *     no C++ exception crosses this boundary;
 *   - all pointer arguments are HOST pointers borrowed for the duration of the call, unless the
 *     name says `_device`;
 *   - a handle is driven by one thread at a time (Send, not Sync in Rust terms);
 *   - one handle owns ONE GPU and one contiguous shard of the particle population; a
 *     multi-GPU filter is `world_size` handles (one per GPU, one per process or per thread)
 *     that call every collective entry point (create / update / step / pose /
 *     map_probability / destroy) in the same order with the same arguments.
 *   - grid cells are addressed `index = row * grid_h + column` with column = x, row = y
 *     (slamrs/slam/src/grid/map.rs:194-204); grids must be square (the reference's index
 *     formula aliases otherwise).
 */
#ifndef SLAMRS_GPU_H
#define SLAMRS_GPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SLAMRS_GPU_ABI_VERSION 1
#define SLAMRS_NCCL_ID_BYTES 128

enum slamrs_status {
    SLAMRS_OK = 0,
    SLAMRS_E_INVALID_ARG = -1,   /* null pointer, zero particles, non-square grid, bad rank ... */
    SLAMRS_E_CUDA = -2,          /* a CUDA runtime call failed; see slamrs_gpu_last_error */
    SLAMRS_E_NCCL = -3,          /* NCCL unavailable or a collective failed */
    SLAMRS_E_OUT_OF_MEMORY = -4, /* device allocation failed */
    SLAMRS_E_NO_DEVICE = -5,     /* no CUDA device: there is NO CPU fallback */
    SLAMRS_E_STAGING = -6,       /* cross-GPU migration needed more free grid slots than exist */
    SLAMRS_E_NOT_LOCAL = -7,     /* debug accessor asked for a particle owned by another rank */
    SLAMRS_E_INTERNAL = -8,
    SLAMRS_E_WINDOW = -9         /* a scan could not be proven to fit a grid's windowed slot (see slot_cells) */
};

enum slamrs_rng_mode {
    SLAMRS_RNG_SHARED_STREAM = 0, /* library draws from the Philox4x32-10 shared stream (DESIGN.md) */
    SLAMRS_RNG_CALLER = 1         /* caller passes the standard-normal draws and the resample uniform */
};

enum slamrs_flags {
    /* use the 32-bit-window ray kernel even where the packed 16-bit-window kernel applies
     * (tests run both; results are identical) */
    SLAMRS_FLAG_GENERIC_RAY_KERNEL = 1,
    /* Strict order of work: integrate the scan into EVERY particle's grid, as the reference does
     * (slam.rs:65-68), instead of only into the grids that survive this step's resampling. The
     * observable state is identical either way (dropped particles are never read again); the
     * default skips the unobservable work. */
    SLAMRS_FLAG_UPDATE_ALL_PARTICLES = 2,
    /* Resampling copies whole grids (W*H cells each), as `Map::clone` does (particle.rs:97-100).
     * The default moves only the informed extent of each grid -- cells outside it are still at
     * the prior in source and destination alike, so the result is identical. Grids whose side is
     * not a multiple of 8 cells always use whole-grid copies. */
    SLAMRS_FLAG_FULL_GRID_COPY = 4,
    /* Multi-GPU only. Exchange the per-particle results with ncclAllGather and synchronise the
     * ranks with NCCL all-reduces. The default fuses the exchange into the likelihood kernel
     * (each record is stored straight into every peer's copy over NVLink) and synchronises through
     * peer-mapped flags, which costs a few microseconds instead of a collective launch. */
    SLAMRS_FLAG_NCCL_EXCHANGE = 8,
    /* Copy every clone when resampling creates it, as `value.clone()` does (particle.rs:97-100).
     * The default defers: a clone shares its source's cells until it is written, i.e. until its
     * particle survives a later resampling and receives a scan -- which, with thousands of particles
     * and a few hundred survivors per step, most clones never do. The observable state is identical.
     * Whole-grid copies (SLAMRS_FLAG_FULL_GRID_COPY) are always eager. */
    SLAMRS_FLAG_EAGER_COPY = 16
};

typedef struct slamrs_gpu_handle slamrs_gpu_handle;

/* Replaces `GridMapSlamConfig` (slam.rs:18-25) plus the placement the YAML cannot carry. */
typedef struct slamrs_gpu_config {
    uint32_t struct_size;  /* = sizeof(slamrs_gpu_config) */
    uint32_t abi_version;  /* = SLAMRS_GPU_ABI_VERSION */
    float pos_x, pos_y;    /* GridMapSlamConfig.position (world position of cell (0,0)'s corner) */
    float resolution;      /* metres per cell */
    uint32_t grid_w;       /* ceil(width / resolution) in f32, map.rs:28-31; see slamrs_gpu_grid_cells */
    uint32_t grid_h;       /* must equal grid_w */
    uint64_t n_particles;  /* TOTAL over all ranks; must be divisible by world_size */
    uint64_t seed;         /* shared-stream key */
    uint32_t rng_mode;     /* enum slamrs_rng_mode */
    int32_t device;        /* CUDA ordinal, -1 = current device */
    uint32_t rank;         /* 0 .. world_size-1 */
    uint32_t world_size;   /* 1 = single GPU */
    uint32_t spare_slots;  /* extra physical grid slots per GPU used to stage grids that migrate
                              between GPUs at resampling; 0 = automatic (none when world_size==1) */
    uint32_t flags;        /* enum slamrs_flags bits, normally 0 */
    uint32_t slot_cells;   /* 0: every particle's slot holds the whole grid. Otherwise a power of two >= 256:
                              a slot holds a slot_cells x slot_cells torus of the grid, enough for the informed
                              extent of one particle's map (everything else is the prior). Memory per particle
                              drops from 4*W*H to 4*slot_cells^2 bytes. Before a grid receives a scan, the step
                              proves that its extent will still fit, conservatively: with reach = ceil(m / resolution)
                              + 6 cells, m the largest |distance| over EVERY beam of the scan, valid or not (a
                              non-finite distance is unbounded; a device-resident scan uses its max_dist), the square
                              of side 2*reach + 1 around the start cell (columns widened to multiples of 8, clipped to
                              the grid) united with the informed extent must fit slot_cells x slot_cells. Otherwise
                              that grid is left as it was and the step reports SLAMRS_E_WINDOW, even where the cells
                              the rays would write fit: one long beam (e.g. an invalid reading at 13 m on 5 cm cells
                              with slot_cells = 512) refuses the step for every particle, and a scan without beams
                              still has reach 6. set_cells refuses an image whose extent, columns widened to
                              multiples of 8, does not fit. */
    float resample_threshold; /* 0 (default): resample after every update, as the reference does (slam.rs:74).
                                 tau in (0, 1]: resample only when the effective number of particles
                                 (particle.rs:59-65) is below tau * N; otherwise every particle stays in place and
                                 carries its normalised weight into the next update (SURVEY.md 8(f)4; not a
                                 reference feature). With tau > 0, N_eff is the reference's strict left fold of
                                 the squared weights, bit for bit, so the decision is the reference's even when
                                 N_eff lies within an ulp of tau * N; at 0 it is a re-associated sum (within 1e-9) */
    uint8_t nccl_id[SLAMRS_NCCL_ID_BYTES]; /* from slamrs_gpu_nccl_unique_id, same on all ranks */
} slamrs_gpu_config;

/* Per-step counters for benchmarks and tests (last completed step). */
typedef struct slamrs_gpu_stats {
    uint64_t step;             /* number of completed updates */
    uint64_t grids_copied;     /* grids copied in the last step: clones made private + eager copies + pulls (D) */
    uint64_t grids_pulled;     /* grids fetched from other GPUs over NVLink */
    uint64_t distinct_sources; /* distinct surviving particles among this rank's new generation */
    uint64_t resample_clamped; /* 1 if a resample index ran past N-1 (the reference would panic) */
    uint64_t counter_saturated;/* cells whose u16 counter hit 65535 in this step */
    uint64_t spilled_cells;    /* ray cell-steps that fell outside the shared-memory window */
    uint64_t window_cells;     /* shared-memory window size used by the ray kernel (cells) */
    uint64_t bytes_per_grid;   /* device bytes of one particle grid */
    uint64_t particles_integrated; /* local particles whose grid received the scan this step */
    uint64_t copy_bytes;       /* bytes the resampling copies read + wrote in this step (device-counted) */
    uint64_t window_overflow;  /* grids whose informed extent would have outgrown a windowed slot (error) */
    uint64_t resample_exact_fallback; /* bit 0 / 1 / 2: the weight sum / the running sum / the sum of squares (only
                                         with resample_threshold > 0) of the last step was folded by a single thread
                                         (NaN, inf or hostile weights; the result is the same) */
    uint64_t resample_fold_rounds;    /* rounds the parallel exact fold needed (1 = proven at once) */
    uint64_t resampled;               /* 1 if the last update resampled (always, unless resample_threshold > 0) */
} slamrs_gpu_stats;

/* ------------------------------------------------------------------ lifecycle */

/* Map::new's grid sizing, map.rs:28-31: `(extent / resolution).ceil() as usize` in f32. */
int slamrs_gpu_grid_cells(float extent, float resolution, uint32_t* out_cells);

/* Fill `out` with a fresh NCCL unique id (call on rank 0, distribute to every rank's config). */
int slamrs_gpu_nccl_unique_id(uint8_t out[SLAMRS_NCCL_ID_BYTES]);

/* GridMapSlam::new, slam.rs:28-43 (Map::new map.rs:26-48, ParticleFilter::new particle.rs:15-28):
 * N particles at Pose::default() with all-prior maps and weight 1/N. Collective when world_size>1. */
int slamrs_gpu_create(const slamrs_gpu_config* cfg, slamrs_gpu_handle** out);

/* Drop. Safe on NULL. A later create in the same process must work (baseui/src/app.rs:121-134). */
void slamrs_gpu_destroy(slamrs_gpu_handle* h);

/* ------------------------------------------------------------------ the step */

/* GridMapSlam::update(&mut self, z: &Observation, u: Odometry), slam.rs:46-75.
 *   angle/dist : `m.angle as f32`, `m.distance as f32` per measurement (map.rs:76-77,121-122)
 *   valid      : Measurement.valid (robot.rs:93)
 *   dist_left / dist_right / wheel_dist : the three Odometry floats (robot.rs:115-123); the two
 *                Normal distributions are derived inside exactly as Odometry::new does (:132-150)
 *   z_draws    : rng_mode CALLER: 2*n_particles standard normals, particle-major
 *                (centre-distance draw, heading draw -- the draw order of robot.rs:175-176);
 *                every rank passes the full array. NULL in SHARED_STREAM mode.
 *   resample_u : rng_mode CALLER: pointer to the uniform [0,1) of particle.rs:84. NULL otherwise.
 * Synchronous: on return the new generation is complete (reference semantics, node.rs:49-57). */
int slamrs_gpu_update(slamrs_gpu_handle* h, const float* angle, const float* dist, const uint8_t* valid,
                      uint32_t n_beams, float dist_left, float dist_right, float wheel_dist,
                      const double* z_draws, const double* resample_u);

/* The same step split for pipelined callers and for device-resident benchmarking:
 * upload_scan copies the observation to the device (async on the handle's stream);
 * step_async enqueues one full SLAM step on the device-resident scan and returns immediately;
 * sync waits for the handle's stream. update() == upload_scan + step_async + sync. */
int slamrs_gpu_upload_scan(slamrs_gpu_handle* h, const float* angle, const float* dist, const uint8_t* valid,
                           uint32_t n_beams);
int slamrs_gpu_step_async(slamrs_gpu_handle* h, float dist_left, float dist_right, float wheel_dist,
                          const double* z_draws, const double* resample_u);
int slamrs_gpu_sync(slamrs_gpu_handle* h);
/* Use an observation that already lives in device memory (caller-owned, must stay valid until
 * the steps that use it have completed). max_dist = an upper bound of |distance| over every beam
 * of the scan, in metres: it sizes the ray kernel's shared-memory window. +inf, NaN or a value <= 0
 * mean "unknown" (pass +inf when the scan may hold non-finite distances): the step then takes the
 * unfused ray update, which is exact for any scan. A bound that some beam exceeds can make the
 * step fail with SLAMRS_E_INTERNAL. */
int slamrs_gpu_set_scan_device(slamrs_gpu_handle* h, const float* angle_device, const float* dist_device,
                               const uint8_t* valid_device, uint32_t n_beams, float max_dist);

/* GridMapSlam::estimated_pose, slam.rs:77-81 -> {x, y, theta}. Reproduces the reference's
 * indexing: particle `max_particle` (argmax BEFORE resampling) of the NEW generation. */
int slamrs_gpu_pose(slamrs_gpu_handle* h, float out_xyt[3]);

/* GridMapSlam::estimated_likelihood, slam.rs:83-88 -> grid_w*grid_h probabilities (f64), the
 * payload of GridMapMessage.data (node.rs:68-72). Collective when world_size>1: every rank calls it
 * (one barrier); a rank that passes a buffer converts the estimate straight out of the owning GPU's
 * pool over NVLink, a rank that passes NULL takes part without receiving the map (the reference has
 * one consumer, node.rs:53-57). */
int slamrs_gpu_map_probability(slamrs_gpu_handle* h, double* out_cells);
/* The same read-out for a pipelined caller (a node that publishes map t while step t+1 runs): the conversion is
 * queued behind the steps issued so far, the copy into out_cells (page-locked host memory, or the copy is not
 * asynchronous) runs on a stream of its own, and the call returns at once; out_cells holds the map once
 * slamrs_gpu_map_wait has returned. Steps issued in between overlap the copy and do not disturb it (the map is
 * converted into one of two device buffers first); at most two read-outs may be pending. Collective like
 * map_probability when world_size>1. */
int slamrs_gpu_map_probability_async(slamrs_gpu_handle* h, double* out_cells);
int slamrs_gpu_map_wait(slamrs_gpu_handle* h);

/* Cheaper forms of the same read-out for consumers that do not need 8 bytes per cell of the whole
 * grid (SURVEY.md 8(f)3; the visualizer converts every cell to an f32 grey level,
 * baseui/src/node/visualize.rs:245-256). map_extent returns the informed extent [x0,x1) x [y0,y1)
 * of the estimate's grid in cells (x0, x1 multiples of 8; all zeros while the map is empty): every
 * cell outside it is exactly at the prior, 0.5. map_window exports the window [x0,x1) x [y0,y1),
 * row-major, as f64, f32 or u8 = round(255 p). Collective when world_size>1 (map_window: out may be NULL
 * on ranks that only take part). */
enum slamrs_map_format { SLAMRS_MAP_F64 = 0, SLAMRS_MAP_F32 = 1, SLAMRS_MAP_U8 = 2 };
int slamrs_gpu_map_extent(slamrs_gpu_handle* h, int32_t out_x0y0x1y1[4]);
int slamrs_gpu_map_window(slamrs_gpu_handle* h, uint32_t format, int32_t x0, int32_t y0, int32_t x1, int32_t y1,
                          void* out);

/* ParticleFilter::number_of_effective_particles, particle.rs:59-65, evaluated on the normalised
 * weights of the last update BEFORE resampling (the reference never calls it; after resampling it
 * is trivially N). N before the first update. */
int slamrs_gpu_effective_particles(slamrs_gpu_handle* h, double* out);

/* Global-localisation-style start (README.md:45 lists it as an idea; SURVEY.md 8(f)4): every particle of this
 * rank's shard gets a pose drawn uniformly over the box {x0, y0, x1, y1} (metres), heading in [-pi, pi), from
 * the shared stream keyed by the config's seed and the GLOBAL particle index (any sharding gives the same
 * population). Maps are untouched. Call before the first update (or any time between updates). */
int slamrs_gpu_init_uniform(slamrs_gpu_handle* h, const float box_x0y0x1y1[4]);

/* ------------------------------------------------------------------ scan production on the device */

/* The simulator's lidar (slamrs/simulator/src/sim.rs:134-159, scene/ray.rs:55-83) evaluated on the
 * device, straight into the handle's scan buffers: n_beams rays at 360/n_beams degree steps from
 * pose {x, y, theta} against n_segments line segments {x1, y1, x2, y2}; rays that hit nothing are
 * dropped, hits beyond scanner_range become invalid measurements at scanner_range. The next
 * step_async consumes it; *out_n (optional) receives the number of measurements. */
int slamrs_gpu_sim_scan(slamrs_gpu_handle* h, const float* segments_xyxy, uint32_t n_segments, const float pose_xyt[3],
                        uint32_t n_beams, float scanner_range, uint32_t* out_n);
/* Copy the device-resident observation back (at most cap measurements; *out_n = how many exist). */
int slamrs_gpu_get_scan(slamrs_gpu_handle* h, float* out_angle, float* out_dist, uint8_t* out_valid, uint32_t cap,
                        uint32_t* out_n);

/* ------------------------------------------------------------------ scan-matching pose refinement */

/* Not in the reference (the slam.rs:60 TODO). Off by default; while it is off the step is unchanged. When it is on,
 * each sampled pose is moved onto its particle's own pre-update grid before the likelihood, by a hill climb on an
 * integer score, bit-exact against the CPU oracle:
 *   S(pose) = sum over valid beams of max((r+1)^2 - (dx^2 + dy^2)) over the occupied cells (counters' log-odds > 0)
 *             at offsets (dx, dy) in [-r, r]^2 of the endpoint's cell (0 when there is none or the endpoint is off
 *             the grid);
 *   for level = 0 .. levels-1 (steps step_xy * 2^-level, step_theta * 2^-level), while moves < max_moves: score
 *   (x+d, y, t), (x-d, y, t), (x, y+d, t), (x, y-d, t), (x, y, t+dt), (x, y, t-dt); move to the first best one if it
 *   scores more than the current pose, else go to the next level.
 * The refined pose replaces the sample, and the motion log-density is recomputed from the old pose to it. The scan is
 * then weighted and integrated at the refined pose. One more kernel per step. */
typedef struct slamrs_gpu_scan_match {
    uint32_t struct_size;   /* = sizeof(slamrs_gpu_scan_match) */
    uint32_t radius;        /* 0..2 cells */
    float step_xy;          /* metres, finite, > 0 */
    float step_theta;       /* radians, finite, > 0 */
    uint32_t levels;        /* 1..8 */
    uint32_t max_moves;     /* 1..1024 */
} slamrs_gpu_scan_match;
/* Takes effect at the next step; NULL turns the matcher off. With world_size > 1 every rank sets the same value before
 * the same step. A localiser handle returns SLAMRS_E_INVALID_ARG. */
int slamrs_gpu_set_scan_match(slamrs_gpu_handle* h, const slamrs_gpu_scan_match* m);
/* Of this rank's particles in the last step: {particles that moved, total moves, poses scored (start poses included),
 * particles that stopped at max_moves}. All zero when the last step ran without the matcher. Synchronises. */
int slamrs_gpu_get_scan_match_stats(slamrs_gpu_handle* h, uint64_t out[4]);

/* ------------------------------------------------------------------ localisation on a loaded map */

/* Monte Carlo localisation: GridMapSlam::update (slam.rs:46-75) with the map held fixed and shared by every particle
 * -- no integration, no per-particle grids (about 100 bytes per particle instead of a grid each). The beam term of
 * each endpoint comes from a per-cell table built on the device at create from the loaded map and a sensor model:
 *   SLAMRS_SENSOR_BEAM_ENDPOINT  the reference's Map::probability_of factor (map.rs:130-141): log(0.9 p + 0.1), 0 for
 *                                p == 0.5 and for endpoints off the grid. Unknown space scores best, so this model
 *                                cannot localise from a uniform start; it is there for parity with the SLAM step.
 *   SLAMRS_SENSOR_LIKELIHOOD_FIELD  log(z_hit exp(-d^2 / (2 sigma^2)) + z_rand), d = distance from the endpoint's cell
 *                                to the nearest cell with p > occupied_above (exact, in cells, times the resolution);
 *                                log(z_rand) off the grid. The model for global localisation. */
enum slamrs_sensor_kind { SLAMRS_SENSOR_BEAM_ENDPOINT = 0, SLAMRS_SENSOR_LIKELIHOOD_FIELD = 1 };
typedef struct slamrs_gpu_sensor_model {
    uint32_t struct_size;    /* = sizeof(slamrs_gpu_sensor_model) */
    uint32_t kind;           /* enum slamrs_sensor_kind */
    float sigma;             /* likelihood field: std. dev. of the hit Gaussian, metres */
    float z_rand;            /* likelihood field: weight of the uniform term, (0, 1); z_hit = 1 - z_rand */
    float occupied_above;    /* likelihood field: obstacle iff p > occupied_above, [0.5, 1) */
} slamrs_gpu_sensor_model;

/* A handle in localiser mode on the grid_w * grid_h probabilities map_probability (index row * grid_h + column, what
 * slamrs_gpu_map_probability writes). Uses position, resolution, grid size, n_particles, seed, rng_mode, device and
 * resample_threshold of cfg; world_size must be 1 and flags, slot_cells and spare_slots 0. Particles start at
 * Pose::default(); place them with init_uniform or set_poses. update / step_async / pose / weights and the other
 * particle accessors work as on a SLAM handle (step_async launches three kernels); the grid accessors (map_*,
 * get_cells, set_cells, get_log_odds, get_extents, get_slots, get_step_history) return SLAMRS_E_INVALID_ARG. */
int slamrs_gpu_create_localizer(const slamrs_gpu_config* cfg, const slamrs_gpu_sensor_model* model,
                                const double* map_probability, slamrs_gpu_handle** out);
/* the localiser's grid_w * grid_h term table (f64, index row * grid_h + column), for tests */
int slamrs_gpu_get_sensor_terms(slamrs_gpu_handle* h, double* out_cells);

/* ------------------------------------------------------------------ introspection (tests, bench) */

const char* slamrs_gpu_last_error(const slamrs_gpu_handle* h); /* never NULL; "" when none */
int slamrs_gpu_get_stats(slamrs_gpu_handle* h, slamrs_gpu_stats* out);
/* cudaStream_t the step runs on, for CUDA-event timing by the caller */
void* slamrs_gpu_stream(slamrs_gpu_handle* h);
/* number of kernels this handle has launched since create */
uint64_t slamrs_gpu_launch_count(const slamrs_gpu_handle* h);

/* Per-phase device timing (CUDA events on the handle's stream). enable, run steps, then read:
 * out_ms[SLAMRS_PHASE_COUNT] = summed milliseconds per phase, *out_steps = steps covered.
 * Reading synchronises the stream and resets the accumulation. */
enum slamrs_phase {
    SLAMRS_PHASE_MOTION_LIKELIHOOD = 0,
    SLAMRS_PHASE_ALL_GATHER = 1,
    SLAMRS_PHASE_RESAMPLE = 2,   /* weights + indices + survivor list + list of shared grids to make private */
    SLAMRS_PHASE_MATERIALIZE = 3,/* separate copies that give surviving clones their own cells (row-major / windowed slots; the
                                    default ray update makes them itself) */
    SLAMRS_PHASE_RAY_UPDATE = 4,
    SLAMRS_PHASE_PULL = 5,       /* join with the side stream (planner; multi-GPU: the NVLink pulls that ran beside the ray
                                    update) + the cross-GPU barrier of the modes that still need one */
    SLAMRS_PHASE_COPY = 6,       /* eager fan-out copies / whole-grid copies, commit */
    SLAMRS_PHASE_COUNT = 7
};
int slamrs_gpu_set_profiling(slamrs_gpu_handle* h, int enabled);
int slamrs_gpu_get_phase_ms(slamrs_gpu_handle* h, double out_ms[SLAMRS_PHASE_COUNT], uint64_t* out_steps);
/* Per-step history (ring of the last 256 steps): for step indices first_step .. first_step+count-1
 * writes SLAMRS_HISTORY_VALUES values per step: {grids_copied, grids_pulled, distinct_sources,
 * source_reads, particles_integrated, copy_bytes, ray_cell_steps, ray_copy_bytes} where source_reads = number of
 * times the copy kernel read a source grid (one read feeds up to 16 destination grids), copy_bytes =
 * bytes the copy kernels really read + wrote, and ray_cell_steps = steps of the reference's ray
 * iterator (ray.rs:83-110) over all rays integrated in that step (0 with the generic ray kernel).  ray_copy_bytes = the part of copy_bytes that the ray update itself moved (a surviving clone's cells are
 * copied by the kernel that integrates its scan). */
#define SLAMRS_HISTORY_VALUES 8
int slamrs_gpu_get_step_history(slamrs_gpu_handle* h, uint64_t first_step, uint32_t count, uint64_t* out_values);

/* current generation, this rank's shard: n_local * {x, y, theta} */
int slamrs_gpu_get_poses(slamrs_gpu_handle* h, float* out_xyt);
int slamrs_gpu_set_poses(slamrs_gpu_handle* h, const float* xyt);
/* the resampler's bookkeeping: physical grid slot of every local particle (n_local entries) and the
 * list of spare slots (*out_n_spare entries; pass a buffer of spare_slots entries, or NULL) */
int slamrs_gpu_get_slots(slamrs_gpu_handle* h, int32_t* out_slot_of, int32_t* out_spare, uint32_t* out_n_spare);
/* last step, all N particles in pre-resample order: normalised and raw (un-normalised) weights */
int slamrs_gpu_get_weights(slamrs_gpu_handle* h, double* out_norm, double* out_raw);
/* last step's resample source index for every new particle (N entries) and the stored argmax */
int slamrs_gpu_get_resample_indices(slamrs_gpu_handle* h, uint32_t* out_idx);
int slamrs_gpu_get_max_particle(slamrs_gpu_handle* h, uint64_t* out);
/* one particle's grid as packed hit counters: low 16 bits = free updates, high 16 = occupied
 * updates; log-odds = n_free*ln(0.3/0.7) + n_occ*ln(0.9/0.1) (map.rs:154-156). `particle` is a
 * GLOBAL logical index and must be owned by this rank. */
int slamrs_gpu_get_cells(slamrs_gpu_handle* h, uint64_t particle, uint32_t* out_cells);
int slamrs_gpu_set_cells(slamrs_gpu_handle* h, uint64_t particle, const uint32_t* cells);
/* the resampler's view of one particle's grid: informed bounding box {x0, y0, x1, y1} (out_box_shift[4] is
 * always 0: slots had a row rotation before they were tiled); per band of 8 slot rows the informed column range x0 | x1 << 16 (0: none),
 * *out_n_bands entries (slot height / 8) -- pass NULL to query the count first */
int slamrs_gpu_get_extents(slamrs_gpu_handle* h, uint64_t particle, int32_t out_box_shift[5], uint32_t* out_bands,
                           uint32_t* out_n_bands);
/* same grid as f64 log-odds (what the reference stores per cell, math.rs:104) */
int slamrs_gpu_get_log_odds(slamrs_gpu_handle* h, uint64_t particle, double* out_cells);

/* ------------------------------------------------------------------ kernel-level test hooks */

/* GridRayIterator (ray.rs:21-110) on the device for n_rays rays in grid coordinates.
 * out_xy holds n_rays * cap * 2 int32 (x, y) pairs, out_count the number of cells each ray
 * visits (may exceed cap; only the first cap are stored). */
int slamrs_gpu_debug_raycast(int device, const float* x0, const float* y0, const float* x1, const float* y1,
                             uint32_t n_rays, uint32_t grid_w, uint32_t grid_h, uint32_t extra_steps,
                             int32_t* out_xy, uint32_t cap, uint32_t* out_count);
/* the device's f32 sin/cos used for poses and endpoints (bit-identical to glibc sinf/cosf) */
int slamrs_gpu_debug_sincos(int device, const float* x, uint32_t n, float* out_sin, float* out_cos);
/* the shared stream evaluated on the device: 2*count normals for particles first.. and the
 * resample uniform of `step` */
int slamrs_gpu_debug_stream(int device, uint64_t seed, uint64_t step, uint64_t first, uint64_t count,
                            double* out_z, double* out_u);

/* normalize_weights, the argmax and the resample indices (particle.rs:40-56, 78-101) for n caller-supplied
 * raw weights and the uniform u01, by the two kernels the step itself runs (k_weights, k_resample_indices).
 * The sums are the reference's strict left folds, reproduced bit for bit (DESIGN.md section 5), so
 * out_idx, out_norm and out_cum (the running sum `c` of particle.rs:85-93 after each weight) equal what
 * the reference computes from the same weights. out_info = {indices clamped to n-1 (the reference would
 * panic), rounds the exact fold needed, chunks resolved by its sequential chain, fallback bits (1: sum,
 * 2: running sum folded by a single thread)}; out_us (optional) = mean device time in microseconds of
 * {k_weights, k_resample_indices} over 20 launches. */
int slamrs_gpu_debug_resample(int device, const double* raw_weights, uint32_t n, double u01, uint32_t* out_idx,
                              uint64_t* out_max_particle, double* out_norm, double* out_cum, uint64_t out_info[4],
                              float out_us[2]);
/* slamrs_gpu_debug_resample with the adaptive-resampling threshold tau (resample_threshold, 0 or in (0, 1]).
 * Also returns (each optional) out_n_eff = the N_eff of particle.rs:59-65 that k_weights computed, out_do_resample
 * = 1 if N_eff < tau * N or tau = 0 (else out_idx is the identity), and out_shape = the launch k_weights used
 * for n: {CTAs in the cluster, threads per CTA, consecutive elements per thread, 1 = elements held in registers /
 * 0 = the generic kernel that re-reads them from global memory}. Bit 2 of out_info[3]: the sum of squares was
 * folded by a single thread (tau > 0 only). */
int slamrs_gpu_debug_resample_adaptive(int device, const double* raw_weights, uint32_t n, double u01, double tau,
                                       uint32_t* out_idx, uint64_t* out_max_particle, double* out_norm, double* out_cum,
                                       uint64_t out_info[4], float out_us[2], double* out_n_eff, uint64_t* out_do_resample,
                                       uint64_t out_shape[4]);

#ifdef __cplusplus
}
#endif
#endif /* SLAMRS_GPU_H */
