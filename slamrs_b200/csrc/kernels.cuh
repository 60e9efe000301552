// Kernel parameter blocks and launch wrappers of the SLAM step. Hand-written sm_100a kernels, no
// tensor cores anywhere (nothing here is a dense contraction); the step is HBM-bound (grid copies)
// with an instruction-bound cell walk in front of it. Definitions:
//
//   kernels_likelihood.cu  k_motion        robot.rs:152-183 (sample, motion pdf)   one thread per particle
//                          k_likelihood    map.rs:113-145 (beam-endpoint likelihood) one warp per particle,
//                                          results stored into every peer GPU; k_peer_barrier
//   kernels_ray.cu         k_ray_update*   map.rs:71-106 + ray.rs:21-110 + map.rs:148-172 (integrate):
//                                          one CTA per surviving particle, shared-memory disc window
//   kernels_scan_match.cu  k_scan_match    scan-matching pose refinement (extension, off by default): one warp
//                                          per particle, between k_motion and k_likelihood
//   kernels_resample.cu    k_weights       particle.rs:40-56, 59-65 + the running sum of :85-91 (8-CTA cluster)
//                          k_resample_indices  particle.rs:78-101 + survivor list;  k_plan  keep / copy lists
//   kernels_copy.cu        k_copy, k_copy_prepare / k_copy_boxed / k_commit_boxes   particle.rs:97-100 clone()
//   kernels_misc.cu        k_export*       slam.rs:83-88 / map.rs:50-52;  k_sim_scan  simulator/src/sim.rs:134-159
//   kernels_localize.cu    k_loc_step      localisation on a loaded map: motion + likelihood, one warp per 32 particles;
//                          k_loc_terms_beam / k_loc_dt_cols / k_loc_dt_rows   sensor-term table at create
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "slam_device.cuh"

namespace slamrs {

// Result of the per-particle motion + likelihood pass, one record per particle of the WHOLE
// population (each rank fills its shard; an all-gather completes the array on every GPU).
struct alignas(8) ParticleResult {
    double weight;        // exp(log p(z|x,m) + log p(x'|x,u)), un-normalised (slam.rs:62,71)
    float x, y, theta;    // pose sampled from the motion model (robot.rs:170-183)
    int32_t slot;         // physical grid slot on the owning GPU (read by other ranks' planners)
};
static_assert(sizeof(ParticleResult) == 24, "ParticleResult is exchanged between GPUs as 24 bytes");

// Device-resident step state shared by the resampling kernels.
struct StepCounters {
    unsigned long long max_particle;     // argmax of the normalised weights, last max wins (particle.rs:40-46)
    unsigned long long n_copies;         // grids this rank writes in this step (local and remote sources)
    unsigned long long n_leaders;        // sub-runs of <= COPY_FAN copies sharing one source read
    unsigned long long n_pulls;          // distinct remote sources this rank copies from in this step
    unsigned long long distinct;         // distinct sources feeding this rank's new generation
    unsigned long long clamped;          // resample index clamped to N-1
    unsigned long long saturated;        // cells that hit the u16 ceiling this step
    unsigned long long spilled;          // ray cell-steps outside the shared-memory window
    unsigned long long staging_short;    // free slots missing for cross-GPU pulls (error)
    long long est_slot;                  // physical slot of new-generation particle max_particle, -1 if remote
    unsigned long long est_owner;        // rank that owns it
    unsigned long long n_spare;          // entries of the persistent spare-slot list
    unsigned long long n_alive;          // local particles whose grid is integrated this step
    unsigned long long copy_bytes;       // bytes read + written by the copy kernels this step
    unsigned long long copy_max_rows;    // tallest region any copy job of this step writes (rows)
    unsigned long long barrier_timeout;  // 1: a peer barrier gave up waiting, 2: a peer destroyed its handle (errors)
    unsigned long long window_overflow;  // grids whose informed extent would outgrow a windowed slot (error)
    unsigned long long est_meta_ptr;     // SlotMeta whose extent the published map has after this step (0: remote)
    unsigned long long n_mat;            // shared grids made private before this step's ray update (copies)
    unsigned long long n_mat_leaders;    // fan-out sub-runs among them
    unsigned long long ray_cell_steps;   // ray-iterator steps integrated this step (packed ray kernel), for the roofline
    unsigned long long ray_copy_bytes;   // bytes of clone copies the ray update read + wrote this step (part of copy_bytes)
    unsigned long long ray_work_head;    // next item of the ray update's work list (popped by its resident CTAs)
    unsigned long long ray_items_front;  // ray work list: clones whose grid a peer GPU pulls in this step (listed first)
    unsigned long long ray_items_back;   // ray work list: slot owners whose grid a peer GPU pulls (first among the owners)
    unsigned long long ray_items_front_local;  // the other clones (behind the pulled ones)
    unsigned long long ray_items_back_local;   // the other slot owners (last)
    unsigned long long fuse_overflow;    // fused ray update: more parked hits than its scratch holds (error; cannot happen by RAY_OCC_PER_RAY_MAX, kernels_ray.cu)
    unsigned long long do_resample;      // k_weights: this step resamples (always 1 unless adaptive resampling is on)
    unsigned long long carry_active;     // the weights of the last step were carried over (it did not resample)
    unsigned long long fold_rounds;      // k_weights: rounds the exact left fold needed (1 = proven at once)
    unsigned long long fold_heads;       // k_weights: chunks resolved by the sequential chain (binade changes)
    unsigned long long fold_fallback;    // k_weights: bit 0 / 1 = the raw-weight sum / the running sum fell back to one thread
    int est_box[4];                      // that extent {x0, y0, x1, y1}; -1 when another rank owns the estimate
    double sum;                          // sum of raw weights (particle.rs:50)
    double n_eff;                        // 1 / sum of squared normalised weights (particle.rs:59-65)
    float est_pose[3];                   // estimated_pose(), slam.rs:77-81
    float pad;
};

// per-step record kept on the device so that a pipelined caller can read, after the fact, how
// many grids each step really moved (the roofline is computed from moved bytes only)
struct StepRecord {
    unsigned long long step, n_copies, n_pulls, distinct, n_leaders, n_alive, copy_bytes, ray_cell_steps, ray_copy_bytes;
};
constexpr uint32_t STEP_HISTORY = 256;
constexpr uint32_t COPY_FAN = 16;   // destinations written per source read in k_copy

struct ScanDevice {
    const float* angle;
    const float* dist;
    const uint8_t* valid;
    uint32_t n_beams;
    // beam order for the ray kernel: indices sorted by decreasing distance, so that the 32 rays of a
    // warp have similar lengths (a warp walks as long as its longest ray). nullptr = scan order.
    // The grid update is order-independent (integer counters), so this changes no result.
    const uint16_t* order;
};
constexpr uint32_t SORT_MAX_BEAMS = 2048;
// order[0..n) = beam indices by decreasing |dist| (NaN last); n <= SORT_MAX_BEAMS
void launch_sort_beams(cudaStream_t stream, const float* dist, uint32_t n_beams, uint16_t* order);

// Per-slot metadata. [x0, x1) x [y0, y1) is the extent (in cells, x0/x1 multiples of 8) of the
// cells of the slot that may be non-zero: everything outside is guaranteed to be zero
// (never-informed cells), which is what lets the resampler move only the informed part of a grid.
// Empty: x1 <= x0. The array lives at the head of the grid pool allocation, so a peer GPU that
// maps the pool sees the extents of the grids it pulls.
struct alignas(32) SlotMeta {
    int x0, y0, x1, y1;
    int pad0, pad1, pad2, pad3;   // (32 bytes: one sector per slot)
};
static_assert(sizeof(SlotMeta) == 32, "SlotMeta is read by peers as 32 bytes");

struct CopyItem {
    const uint32_t* src;  // may be a peer-mapped pointer (grid on another GPU)
    uint32_t* dst;
    const SlotMeta* src_meta;  // extent of the source grid (peer-mapped for a pull)
    SlotMeta* dst_meta;        // extent of the destination slot (what it held before / holds after)
    const uint32_t* src_bands; // band extents of the source grid (peer-mapped for a remote source)
    uint32_t* dst_bands;       // band extents of the destination slot
};

// One work item of the ray update: a surviving local particle, its slot and the slot whose cells it
// logically holds (root != slot: a clone that k_ray_update_half makes private while it integrates the scan)
struct RayItem {
    uint32_t particle;
    int32_t slot, root;
    int32_t old_y0, old_y1;   // clone: rows [old_y0, old_y1) the slot's previous tenant had informed (to be cleared)
    uint32_t pad;
};
// Work lists of the fused ray update, filled by k_resample_indices: clones first (counters->ray_items_front of
// them), then the particles that own their slot (counters->ray_items_back); readers[root]++ per clone (zeroed by
// the caller); every listed clone's alias entry becomes the identity and counters->n_mat counts them.
// clones == nullptr: plain survivor list (alive_list) instead.
struct RayLists {
    RayItem* clones;
    RayItem* owners;
    const int32_t* slot_of;
    int32_t* alias_of;
    uint32_t* readers;
    SlotMeta* meta;
    uint32_t n_local;        // capacity of clones[] and of owners[]: pulled items fill them from the front, the others from the back
    uint32_t mark_remote;    // world > 1: RayItem::pad = 1 for a particle that a new particle of ANOTHER rank selects (that
                             // rank pulls the grid in this step: listed first, and the ray update signals its completion)
};
// work item k of the lists above: pulled clones, other clones, pulled owners, other owners
__device__ __forceinline__ RayItem ray_item_at(const RayItem* __restrict__ clones, const RayItem* __restrict__ owners,
                                               uint32_t n_local, const StepCounters* counters, unsigned long long k) {
    const unsigned long long n_rc = counters->ray_items_front, n_lc = counters->ray_items_front_local;
    if (k < n_rc) return clones[k];
    k -= n_rc;
    if (k < n_lc) return clones[n_local - 1u - k];
    k -= n_lc;
    const unsigned long long n_ro = counters->ray_items_back;
    if (k < n_ro) return owners[k];
    return owners[n_local - 1u - (k - n_ro)];
}
// ---- launch wrappers (all asynchronous on `stream`) ----
// scan-matching pose refinement (slamrs_gpu_scan_match), between k_motion and k_likelihood
struct ScanMatchParams {
    uint32_t radius;
    float step_xy, step_theta;
    uint32_t levels, max_moves;
};
void launch_motion_likelihood(cudaStream_t stream, MapGeom geom, OdomModel od, ScanDevice scan,
                              const float* pose_cur, const int32_t* slot_of, const int32_t* alias_of /* may be null */,
                              const uint32_t* cells,
                              const SlotMeta* meta, size_t cells_per_grid, ParticleResult* results, uint32_t first_particle,
                              uint32_t n_local, const double* z_draws, uint64_t seed, uint64_t step,
                              const double* term_table /* LK_TABLE_NF x LK_TABLE_NO, launch_fill_term_table */,
                              float2* valid_beams /* scratch: n_beams entries */, uint32_t* n_valid /* scratch */,
                              const double* carry /* adaptive resampling: carried weights (n_total), else null */,
                              const StepCounters* counters,
                              ParticleResult* const* peer_results /* null: no fused exchange */,
                              uint32_t peer_offset /* records in front of this step's generation */, uint32_t rank,
                              uint32_t world, uint32_t* zero_words /* n_zero words that k_motion clears (may be null with 0) */,
                              uint32_t n_zero, const ScanMatchParams* match /* null: no scan matching */,
                              uint2* match_stats /* with match: n_local x {moves, poses scored} */);
void launch_fill_term_table(cudaStream_t stream, double* table);
void launch_scan_match(cudaStream_t stream, MapGeom geom, ScanMatchParams mp, OdomModel od, const float* pose_cur,
                       const int32_t* alias_of /* may be null */, const uint32_t* cells, const SlotMeta* meta,
                       size_t cells_per_grid, ParticleResult* results, uint32_t first_particle, uint32_t n_local,
                       const float2* valid_beams, const uint32_t* n_valid,
                       uint2* stats /* n_local x {moves, poses scored} */);
constexpr uint32_t PEER_MAX_WORLD = 64;
void launch_peer_barrier(cudaStream_t stream, unsigned long long* const* peer_flags, unsigned long long* my_flags,
                         uint32_t rank, uint32_t world, unsigned long long epoch, unsigned long long timeout_ns,
                         StepCounters* counters);
void launch_peer_goodbye(cudaStream_t stream, unsigned long long* const* peer_flags, unsigned long long* my_flags,
                         uint32_t rank, uint32_t world, unsigned long long timeout_ns, StepCounters* counters);

// the fused path applies (packed window kernel, whole-grid tiled slots)
bool ray_update_can_fuse(const MapGeom& geom, uint32_t n_beams, size_t cells_per_grid, bool force_generic, int radius_cells);
size_t ray_spill_scratch_words(int num_sms);
size_t ray_half_xchg_bytes();               // per surviving particle: what its lower half hands to its upper half
int ray_trace(unsigned long long* out18);   // tuning builds (-DSLAMRS_RAY_TRACE): cycles per phase, summed over CTAs   // scratch of the fused path (uint32 words)
// returns the shared-memory window size in cells through *window_cells
// alive_list / counters->n_alive select the local particles to integrate (see launch_mark_alive); with the work
// lists of RayLists (clones, owners) the half-particle kernel fuses the clones' copies into its write-back (readers /
// done: per-slot counters, zeroed by the caller before launch_resample_indices)
cudaError_t launch_ray_update(cudaStream_t stream, MapGeom geom, ScanDevice scan, const ParticleResult* results,
                              uint32_t first_particle, uint32_t n_local, const uint32_t* alive_list,
                              const RayItem* clones, const RayItem* owners, const uint32_t* readers, uint32_t* done,
                              uint32_t* xflag /* per work item, zeroed by the caller */, void* xchg /* n_local * ray_half_xchg_bytes() */,
                              uint32_t* spill_scratch,
                              const int32_t* slot_of, uint32_t* cells, SlotMeta* meta, uint32_t* bands,
                              size_t cells_per_grid, int radius_cells, StepCounters* counters,
                              uint64_t* window_cells, bool force_generic, int num_sms,
                              uint32_t* xdone /* per work item, zeroed by the caller */,

                              uint32_t signal_epoch /* != 0 (half-item kernel only): every integrated slot's SlotMeta::pad0
                                                       receives it once both halves are in place (peers that pull the slot wait for it) */);

// k_weights' launch for a population: a cluster of `cluster` CTAs of `threads` threads, each thread folding `chunk`
// consecutive elements, held in registers (regs) or re-read from global memory (the generic kernel)
struct WeightsShape { uint32_t cluster, threads, chunk; bool regs; };
WeightsShape weights_shape(uint32_t n_total);
// fold_scratch: weights_scratch_doubles() doubles
// resample_tau > 0: counters->do_resample = N_eff < tau * N (adaptive resampling; N_eff from the reference's strict
// left fold of the squares), else 1
void launch_weights(cudaStream_t stream, const ParticleResult* results, uint32_t n_total, double* w_norm,
                    double* cum, double* fold_scratch, double resample_tau, StepCounters* counters);
size_t weights_scratch_doubles();
int weights_trace(long long* out64);   // tuning builds (-DSLAMRS_FOLD_TRACE): clock stamps of the last k_weights

void launch_resample_indices(cudaStream_t stream, const ParticleResult* results, const double* cum,
                             uint32_t n_total, const double* u01_caller, uint64_t seed, uint64_t step,
                             uint32_t* idx, float* pose_next, uint32_t first_particle, uint32_t n_local,
                             bool build_alive /* also list the surviving local particles */,
                             uint32_t* alive_list, RayLists ray, const double* w_norm, double* carry /* may be null */,
                             StepCounters* counters);

struct PlanArgs {
    const ParticleResult* results;  // N, after the all-gather (carries every particle's physical slot)
    const uint32_t* idx;       // N resample sources
    uint32_t n_total, n_local, rank, world;
    const int32_t* slot_old;   // n_local
    int32_t* slot_new;         // n_local
    int32_t* keep;             // n_local scratch
    int32_t* need;             // n_local scratch
    int32_t* free_list;        // n_local + n_spare_cap scratch
    int32_t* spare_list;       // persistent list of free physical slots beyond the live set
    uint32_t n_spare_cap;
    CopyItem* copies;          // n_local
    uint32_t* leaders;         // n_local: positions in copies[] that start a fan-out sub-run
    uint32_t* cells;           // local pool base
    size_t cells_per_grid;
    uint32_t* const* peer_cells;        // world pointers to each rank's pool (device array), may be null when world==1
    SlotMeta* meta;                     // local per-slot extents
    SlotMeta* const* peer_meta;         // world pointers to each rank's extents, may be null when world==1
    uint32_t* bands;                    // local per-slot band extents, n_bands entries per slot
    uint32_t* const* peer_bands;        // world pointers to each rank's band extents
    uint32_t n_bands;
    StepCounters* counters;
    StepRecord* history;       // STEP_HISTORY entries, slot = step % STEP_HISTORY
    unsigned long long step;
    bool staged;               // working arrays in shared memory (plan_can_stage)
    // Shared grids (deferred copies). alias_of[slot] = the slot whose cells `slot` logically holds:
    // itself for a private grid, the source's slot for a clone that has not been written since
    // resampling created it. With `defer` the planner turns every further use of a source into such
    // an alias instead of a copy (only the first use of a REMOTE source is copied, over NVLink);
    // k_materialize_list makes a shared grid private when its particle is about to be written.
    int32_t* alias_of;         // n_local + n_spare_cap
    bool defer;
};
void launch_plan(cudaStream_t stream, const PlanArgs& a);
// Shared grids that are about to be written (local particles selected by the index vector, or all
// of them): one CopyItem (root slot -> the particle's own slot) each, in particle order, fan-out
// leaders as in k_plan; the particles' alias entries become the identity. Counts go to
// counters->n_mat / n_mat_leaders. idx == nullptr: every local particle (also used to un-share
// everything before a grid is overwritten from the host).
void launch_materialize_list(cudaStream_t stream, const uint32_t* idx, uint32_t n_total, uint32_t first_particle,
                             uint32_t n_local, const int32_t* slot_of, int32_t* alias_of, uint32_t* cells,
                             size_t cells_per_grid, SlotMeta* meta, uint32_t* bands, uint32_t n_bands, CopyItem* items,
                             uint32_t* leaders, uint32_t* roots_scratch /* n_local */, StepCounters* counters);
bool plan_can_stage(uint32_t n_local, uint32_t n_spare_cap);

// the same for the particles of the survivor list (counters->n_alive entries): unordered, no fan-out grouping
void launch_materialize_alive(cudaStream_t stream, const uint32_t* alive_list, uint32_t n_local, const int32_t* slot_of,
                              int32_t* alias_of, uint32_t* cells, size_t cells_per_grid, SlotMeta* meta, uint32_t* bands,
                              uint32_t n_bands, CopyItem* items, StepCounters* counters);

// local particles that appear in the index vector (their grid survives resampling); all_particles
// lists every local particle instead (reference order of work)
void launch_mark_alive(cudaStream_t stream, const uint32_t* idx, uint32_t n_total, uint32_t first_particle,
                       uint32_t n_local, bool all_particles, uint32_t* alive_list, StepCounters* counters);

// copies[0..*n_items) full grids; n_items is read on the device
// leaders == nullptr: plain item-by-item copy
void launch_copy(cudaStream_t stream, const CopyItem* items, const uint32_t* leaders,
                 const unsigned long long* n_items, const unsigned long long* n_leaders, size_t cells_per_grid,
                 int num_sms);

// format: 0 = f64, 1 = f32, 2 = u8; [x0, x1) x [y0, y1) is the exported window of the grid
void launch_export(cudaStream_t stream, const uint32_t* cells, const SlotMeta* meta, size_t cells_per_grid,
                   const StepCounters* counters, MapGeom geom, int x0, int y0, int x1, int y1, int format, void* out);
void launch_estimate_extent(cudaStream_t stream, const SlotMeta* meta, const StepCounters* counters, int* out4);
void launch_publish_counters(cudaStream_t stream, const StepCounters* counters, StepCounters* host_mirror);
// one slot's grid in logical order: f64 log-odds (as_log_odds) or the raw packed counters
void launch_export_slot(cudaStream_t stream, const uint32_t* grid, const SlotMeta* slot_meta, MapGeom geom,
                        bool as_log_odds, void* out);

void launch_import_slot(cudaStream_t stream, const uint32_t* image, uint32_t* grid, SlotMeta m, MapGeom geom);
void launch_init_slots(cudaStream_t stream, int32_t* slot_of, uint32_t n_local, int32_t* spare_list, uint32_t n_spare,
                       StepCounters* counters, uint32_t rank, SlotMeta* meta, int32_t* alias_of);

// extent-limited copies: only the informed part of each source grid moves, and the part of the
// destination slot's previous content that the source does not cover is cleared
void launch_copy_boxed(cudaStream_t stream, const CopyItem* items, const uint32_t* leaders,
                       const unsigned long long* n_items, const unsigned long long* n_leaders, uint32_t max_items,
                       void* jobs /* max_items * copy_job_bytes() of scratch */, MapGeom geom,
                       StepCounters* counters, int num_sms, bool short_list = false /* a few hundred items: one wave of CTAs */,
                       uint32_t wait_epoch = 0 /* != 0: a job waits until its source's SlotMeta::pad0 holds it (set by the
                                                  owner's ray update, launch_ray_update's signal_epoch) */,
                       unsigned long long timeout_ns = 0);
size_t copy_job_bytes();
// the same for a short list of REMOTE sources, one CTA per job, each job waiting for its own source (see k_pull)
void launch_pull(cudaStream_t stream, const CopyItem* items, const uint32_t* leaders, const unsigned long long* n_items,
                 const unsigned long long* n_leaders, uint32_t max_items, MapGeom geom, StepCounters* counters, int num_sms,
                 uint32_t wait_epoch, unsigned long long timeout_ns, const SlotMeta* meta_base /* this GPU's slots */,
                 const uint32_t* readers, const uint32_t* done /* the ray update's per-slot reader counts: a destination
                                                                  that clones still read as their root is written after them */);
// after a copy kernel: every destination slot now has its source's extent. With `record` the
// step's moved bytes are also written into the history ring (last copy launch of a step).
// `realign` = extent copy (the copy kernel wrote the band tables); otherwise (whole-grid copies move rows
// verbatim) the band tables are copied here
void launch_commit_boxes(cudaStream_t stream, const CopyItem* items, const unsigned long long* n_items, uint32_t max_items,
                         MapGeom geom, bool realign, StepCounters* counters, StepRecord* record,
                         StepCounters* host_mirror = nullptr /* the step's last kernel: also leaves the counters in the host's
                                                                page-locked mirror */);
// add the bytes of a full-grid copy launch to counters->copy_bytes
void launch_account_full_copy(cudaStream_t stream, const unsigned long long* n_items, const unsigned long long* n_leaders,
                              size_t bytes_per_grid, StepCounters* counters);
// poses of the local shard drawn uniformly over a box (slamrs_stream::uniform_pose)
void launch_init_uniform(cudaStream_t stream, uint64_t seed, uint32_t first_particle, uint32_t n_local, float x0, float y0,
                         float x1, float y1, float* pose);
// simulator lidar into device scan buffers; out_count_maxbits must be zeroed before the launch
void launch_sim_scan(cudaStream_t stream, const float* segments, uint32_t n_seg, float px, float py, float ptheta,
                     uint32_t n_beams, float scanner_range, float* angle, float* dist, uint8_t* valid,
                     uint32_t* out_count_maxbits);
cudaError_t configure_kernels();  // per-device function attributes; call once after cudaSetDevice

// localiser (kernels_localize.cu): the per-cell sensor-term table of a loaded w x w probability map (field = 0: the
// reference's beam-endpoint model; 1: likelihood field, `scratch` = w*w uint32 for its distance transform), and one
// step's motion + likelihood over the whole population into results[0, n) (slot = -1)
cudaError_t launch_loc_terms(cudaStream_t stream, const double* prob, uint32_t w, int field, float sigma, float z_rand,
                             float occupied_above, float res, uint32_t* scratch, double* terms);
void launch_loc_step(cudaStream_t stream, MapGeom geom, OdomModel od, ScanDevice scan, const float* pose_cur,
                     ParticleResult* results, uint32_t n, const double* z_draws, uint64_t seed, uint64_t step,
                     const double* terms, double outside, const double* carry /* adaptive resampling, else null */,
                     const StepCounters* counters);

// test hooks
void launch_debug_raycast(cudaStream_t stream, const float* x0, const float* y0, const float* x1, const float* y1,
                          uint32_t n_rays, uint32_t gw, uint32_t gh, uint32_t extra, int32_t* out_xy, uint32_t cap,
                          uint32_t* out_count);
void launch_debug_sincos(cudaStream_t stream, const float* x, uint32_t n, float* s, float* c);
void launch_debug_stream(cudaStream_t stream, uint64_t seed, uint64_t step, uint64_t first, uint64_t count, double* z,
                         double* u);

}  // namespace slamrs
