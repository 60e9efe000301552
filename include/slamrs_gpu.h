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
    SLAMRS_FLAG_EAGER_COPY = 16,
    /* Issue every step as the serial kernel sequence: stream events fork the planner off and join it, a separate
     * kernel commits the step, and profiling records events between the phases. By default a single-GPU step on a
     * device-resident scan (slamrs_gpu_set_scan_device) with the fused ray update chains its kernels instead: the
     * ray update's last CTA waits for the planner on the device and commits the step, and profiling reads timestamps
     * the kernels take. Results are identical either way. */
    SLAMRS_FLAG_SERIAL_STEPS = SLAMRS_FLAG_EAGER_COPY << 1   /* = 32 */
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
 *   z_draws    : rng_mode CALLER: 2*n_particles standard normals, particle-major (a localiser: 2*N_t, two per
 *                particle of its current generation, see slamrs_gpu_set_kld)
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
 * is trivially N). N before the first update. A localiser: over the last step's N_t particles. */
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
 * particle accessors work as on a SLAM handle (step_async launches three kernels, four with recovery, one more with
 * KLD-sampling; the particle accessors' sizes follow the population, see slamrs_gpu_set_kld); the grid accessors (map_*,
 * get_cells, set_cells, get_log_odds, get_extents, get_slots, get_step_history) return SLAMRS_E_INVALID_ARG. */
int slamrs_gpu_create_localizer(const slamrs_gpu_config* cfg, const slamrs_gpu_sensor_model* model,
                                const double* map_probability, slamrs_gpu_handle** out);
/* the localiser's grid_w * grid_h term table (f64, index row * grid_h + column), for tests */
int slamrs_gpu_get_sensor_terms(slamrs_gpu_handle* h, double* out_cells);

/* Recovery from kidnapping and false convergence: augmented MCL (Probabilistic Robotics, Table 8.3; ROS AMCL's
 * recovery_alpha_slow / recovery_alpha_fast), bit-exact against the CPU oracle. Off by default; while it is off a
 * localiser step is unchanged (three launches, the same bits). When it is on, every step does the following after
 * k_resample_indices, in one more launch (k_loc_recover):
 *   1. w_avg = sum / N, with sum the strict left fold of this step's raw weights (particle.rs:50, motion term
 *      included), by __ddiv_rn; nothing below is contracted.
 *   2. If sum is not finite, the state stays as it is and p = 0. Otherwise
 *        w_slow = (w_slow == 0) ? w_avg : w_slow + alpha_slow * (w_avg - w_slow)
 *        w_fast = (w_fast == 0) ? w_avg : w_fast + alpha_fast * (w_avg - w_fast)
 *        p = (w_slow > 0) ? max(0, 1 - w_fast / w_slow) : 0, NaN mapped to 0.
 *   3. The free cells are the cells of the loaded map with p < 0.5, in ascending cell index (row * grid_h + column),
 *      listed once at create (4 bytes per free cell).
 *   4. Draws from the shared stream keyed by the config seed, in both RNG modes (CALLER mode externalises only the
 *      reference's own draws). For new particle m at step s, Philox counters (m, s lo32, s hi32, d):
 *        d = 4: decision u_d = u53(a0, a1), cell u_c = u53(a2, a3);  d = 5: u_x = u53(b0, b1), u_y = u53(b2, b3);
 *        d = 6: u_t = u53(c0, c1).
 *   5. Particle m is replaced iff u_d < p, by cell free[min(n_free - 1, (uint32)(u_c * n_free))] at column col and
 *      row row: x = (float)(pos_x + (col + u_x) * res), y = (float)(pos_y + (row + u_y) * res),
 *      theta = (float)(-pi + u_t * 2pi), in f64 with pos_x, pos_y and res the config's f32 values.
 *   6. The estimate (estimated_pose: the resampled pose of max_particle), the indices and the weights are the ones
 *      resampling recorded: an injected particle never becomes the estimate in the step that creates it.
 * The cost on a B200 and the behaviour after a kidnapping are in DESIGN.md section 11.1. */
typedef struct slamrs_gpu_recovery {
    uint32_t struct_size;   /* = sizeof(slamrs_gpu_recovery) */
    uint32_t pad;
    double alpha_slow;      /* (0, alpha_fast) */
    double alpha_fast;      /* (alpha_slow, 1] */
} slamrs_gpu_recovery;
/* Localiser only; NULL turns recovery off; setting it resets w_slow and w_fast; takes effect at the next step.
 * Returns SLAMRS_E_INVALID_ARG on a SLAM handle, with resample_threshold > 0 (carried weights put the raw sum on
 * another scale), on a map without free cells, for alphas outside the ranges above and on a struct_size mismatch. */
int slamrs_gpu_set_recovery(slamrs_gpu_handle* h, const slamrs_gpu_recovery* r);
/* Last step: {w_slow, w_fast, p_inject} and the number of particles injected (out_injected may be NULL); all zero
 * when the last step ran without recovery. Synchronises. */
int slamrs_gpu_get_recovery_state(slamrs_gpu_handle* h, double out[3], uint64_t* out_injected);

/* Adaptive population: KLD-sampling (Fox 2003; ROS AMCL's min_particles / max_particles / kld_err / kld_z), bit-exact
 * against the CPU oracle. Off by default; while it is off a localiser step is unchanged (three launches, four with
 * recovery, the same bits) and draws n_particles new particles. cfg.n_particles is the capacity C: every buffer is
 * sized for it at create. The population N_t is the size of the current generation; it starts at C. A step with
 * KLD-sampling on:
 *   1. k = the number of distinct bins occupied by the N_t poses the step starts from (what the previous step,
 *      recovery included, or init_uniform / set_poses left). A pose's cell is the one the likelihood gives a beam
 *      endpoint at (x, y) (world_to_grid, is_valid, `as usize`); heading bin: t = fmod((double)theta, 2pi), t += 2pi
 *      if t < 0, h = min(theta_bins - 1, (uint32)((t * theta_bins) / 2pi)) for 0 <= t < 2pi, else 0 (NaN, inf), in
 *      f64 with 2pi = 0x1.921fb54442d18p+2. Bin ((row / bin_cells) * nbx + column / bin_cells) * theta_bins + h with
 *      nbx = ceil(grid_w / bin_cells); every pose off the grid falls into the one bin nbx * nby * theta_bins.
 *   2. N_{t+1} = n_min for k <= 1; otherwise, in f64 in AMCL's order (pf_resample_limit), uncontracted:
 *      b = 2 / (9 (k - 1)), x = 1 - b + sqrt(b) z, n = (((k - 1) / (2 err)) x) x x, N_{t+1} = clamp(ceil(n), n_min,
 *      n_max), n_max for a non-finite n or one >= n_max.
 *   3. Motion, likelihood and weights over the N_t particles, as without KLD-sampling.
 *   4. M = N_{t+1} draws (particle.rs:78-101 with M wherever N counts draws: r = U * 1.0 / M, u_m = r + (m - 1) * 1.0
 *      / M); the walk over the running sum of the N_t normalised weights and its clamp at N_t - 1 are unchanged.
 *   5. The estimate is new particle floor(max_particle * M / N_t) (64-bit integers), the same cumulative-mass position
 *      as the reference's new[max_particle].
 *   6. Recovery (if on) averages sum / N_t and injects over the M new particles.
 * The size of a step lags AMCL's by one: AMCL counts the bins of the set it draws and stops once the bound is met;
 * here a step draws what the bins of the set it starts from demand (see DESIGN.md section 11.2).
 * One more kernel in front of the step (k_loc_kld: four launches, five with recovery). The host waits for it, so
 * step_async on a handle with KLD-sampling on returns only once that kernel (not the step) has completed.
 * Sizes of the particle accessors on a localiser: get_poses, set_poses and init_uniform use N (the current
 * generation); get_weights and effective_particles the last step's N_t; get_resample_indices its M; a CALLER-mode
 * z_draws holds 2 N_t normals. */
typedef struct slamrs_gpu_kld {
    uint32_t struct_size;   /* = sizeof(slamrs_gpu_kld) */
    uint32_t n_min;         /* 1 <= n_min <= n_max */
    uint32_t n_max;         /* <= n_particles (the capacity) */
    uint32_t pad;
    double err;             /* finite, (0, 1] */
    double z;               /* finite, >= 0: the upper (1 - delta) quantile of the standard normal */
    uint32_t bin_cells;     /* >= 1: grid cells per bin side */
    uint32_t theta_bins;    /* 1..3600 */
} slamrs_gpu_kld;
/* Localiser only; takes effect at the next step; NULL turns it off (the next step then draws n_particles from N_t,
 * and every step after it is the fixed-size step). Returns SLAMRS_E_INVALID_ARG on a SLAM handle, with
 * resample_threshold > 0 (carried weights assume a fixed population), for fields outside the ranges above, for a bin
 * bitmap of more than 2^28 bits and on a struct_size mismatch. */
int slamrs_gpu_set_kld(slamrs_gpu_handle* h, const slamrs_gpu_kld* k);
/* Last step: {N_t particles weighted, k occupied bins, N_{t+1} particles drawn}; all zero when it ran without
 * KLD-sampling. Synchronises. */
int slamrs_gpu_get_kld_state(slamrs_gpu_handle* h, uint64_t out[3]);
/* The size of the current generation: the localiser's population N (n_particles until KLD-sampling changes it); a SLAM
 * handle's n_local. */
int slamrs_gpu_get_population(slamrs_gpu_handle* h, uint64_t* out);

/* Pose hypotheses: clusters of the localiser's current generation with their mean and covariance (ROS AMCL's
 * pf_cluster_stats and the estimate it publishes). Computed on the device on request; DESIGN.md section 11.3.
 *   1. Input: the N poses get_poses returns (the previous step's resampled, injected set, or what init_uniform /
 *      set_poses left), each of weight 1/N. The call is enqueued behind any step_async and synchronises once. It
 *      changes no filter state: poses, weights, indices, estimate, recovery and KLD state, and the launches of the
 *      steps are those of a handle that never calls it.
 *   2. A pose is excluded if any of x, y, theta is not finite or its cell is off the grid (the likelihood's is_valid);
 *      excluded poses are counted in n_excluded and belong to no cluster and not to `overall`.
 *   3. A pose's bin is KLD-sampling's (slamrs_gpu_set_kld, item 1) with these bin_cells and theta_bins:
 *      ((row / bin_cells) * nbx + column / bin_cells) * theta_bins + h.
 *   4. Two occupied bins are adjacent when their (bx, by) differ by at most 1 each and their heading bins differ by at
 *      most 1 modulo theta_bins (AMCL's 3x3x3 neighbourhood, except that the heading wraps: a cloud facing +-pi is one
 *      cluster). A cluster is a connected component of occupied bins; its label is the smallest bin id in it.
 *   5. Clusters are ranked by count (descending), then label (ascending); out_clusters[0, min(K, n_clusters)) receives
 *      the first ones, the rest of its K entries are zeroed. Entry 0 is the estimate AMCL publishes.
 *   6. Moments of each reported cluster and of `overall`, in f64 from the widened f32 coordinates: mean x, y = sums /
 *      count; S = sum sin(theta), C = sum cos(theta); mean theta = atan2(S, C); var_theta = -2 ln(sqrt(S^2 + C^2) /
 *      count). The covariance is centred, in a second pass over the poses: cov_xy = sum (x - mean x)(y - mean y) / count
 *      (AMCL computes E[xy] - E[x]E[y] in one pass). No theta-x or theta-y covariance, as in AMCL. A set without poses
 *      (every pose excluded) reports all zeros.
 *   7. The integer outputs (n_bins, n_clusters, counts, labels, order) are exact; the f64 moments are sums folded in a
 *      fixed order (no floating-point atomics), so every call on the same poses returns the same bits.
 * Returns SLAMRS_E_INVALID_ARG on a SLAM handle, for a NULL c, out or out_clusters, for fields outside the ranges
 * below, for a bin space nbx * nby * theta_bins above 2^28 and on a struct_size mismatch. The device scratch (about
 * 17 bytes per particle of capacity plus 2 bits per bin, at most) is allocated by the first call and kept until destroy. */
typedef struct slamrs_gpu_clustering {
    uint32_t struct_size;   /* = sizeof(slamrs_gpu_clustering) */
    uint32_t bin_cells;     /* >= 1: grid cells per bin side */
    uint32_t theta_bins;    /* 1..3600 */
    uint32_t max_clusters;  /* K, 1..64: clusters reported */
} slamrs_gpu_clustering;

typedef struct slamrs_gpu_pose_cluster {
    uint64_t count;          /* poses in the cluster */
    uint64_t label;          /* smallest bin id in the cluster */
    double weight;           /* count / N */
    double mean[3];          /* x, y (m), theta = atan2(S, C) in (-pi, pi] */
    double cov_xx, cov_xy, cov_yy;  /* centred, divided by count */
    double var_theta;        /* -2 ln(R), R = sqrt(S^2 + C^2) / count (AMCL's cov[2][2]) */
} slamrs_gpu_pose_cluster;

typedef struct slamrs_gpu_pose_stats {
    uint64_t n_poses;        /* N, the current generation */
    uint64_t n_excluded;     /* off the grid or a non-finite component */
    uint64_t n_bins;         /* distinct occupied bins */
    uint64_t n_clusters;     /* all clusters, not only the K reported */
    slamrs_gpu_pose_cluster overall;  /* every non-excluded pose as one set (label 0) */
} slamrs_gpu_pose_stats;

int slamrs_gpu_pose_clusters(slamrs_gpu_handle* h, const slamrs_gpu_clustering* c, slamrs_gpu_pose_stats* out,
                             slamrs_gpu_pose_cluster* out_clusters /* K entries */);

/* ------------------------------------------------------------------ introspection (tests, bench) */

const char* slamrs_gpu_last_error(const slamrs_gpu_handle* h); /* never NULL; "" when none */
int slamrs_gpu_get_stats(slamrs_gpu_handle* h, slamrs_gpu_stats* out);
/* cudaStream_t the step runs on, for CUDA-event timing by the caller */
void* slamrs_gpu_stream(slamrs_gpu_handle* h);
/* number of kernels this handle has launched since create */
uint64_t slamrs_gpu_launch_count(const slamrs_gpu_handle* h);

/* Per-phase device timing. enable, run steps, then read:
 * out_ms[SLAMRS_PHASE_COUNT] = summed milliseconds per phase, *out_steps = steps covered.
 * Reading synchronises the stream and resets the accumulation. The serial step sequence (SLAMRS_FLAG_SERIAL_STEPS)
 * records CUDA events between its phases; a chained step (see that flag) takes %globaltimer stamps inside its
 * kernels instead, which leaves its kernel chain intact. There RAY_UPDATE is the ray kernel's own span, PULL the
 * wait of its last CTA for the planner, COPY the commit; phases of overlapping kernels may overlap, and a phase that
 * another one hides counts 0. */
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

/* current generation, this rank's shard: n_local * {x, y, theta} (a localiser: N, see slamrs_gpu_get_population) */
int slamrs_gpu_get_poses(slamrs_gpu_handle* h, float* out_xyt);
int slamrs_gpu_set_poses(slamrs_gpu_handle* h, const float* xyt);
/* the resampler's bookkeeping: physical grid slot of every local particle (n_local entries) and the
 * list of spare slots (*out_n_spare entries; pass a buffer of spare_slots entries, or NULL) */
int slamrs_gpu_get_slots(slamrs_gpu_handle* h, int32_t* out_slot_of, int32_t* out_spare, uint32_t* out_n_spare);
/* last step, all N particles in pre-resample order: normalised and raw (un-normalised) weights (a localiser: N_t) */
int slamrs_gpu_get_weights(slamrs_gpu_handle* h, double* out_norm, double* out_raw);
/* last step's resample source index for every new particle (N entries; a localiser: M) and the stored argmax */
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
