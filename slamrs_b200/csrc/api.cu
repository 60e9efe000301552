// C ABI of the B200-native grid SLAM step (see include/slamrs_gpu.h).
// Host side: owns device state, sequences the kernels on one stream per GPU, talks NCCL for
// the weight/pose all-gather and maps peer grid pools for cross-GPU migration.
#include "../../include/slamrs_gpu.h"

#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <unistd.h>

#include <algorithm>
#include <new>
#include <string>
#include <vector>

#include "comm.h"
#include "kernels.cuh"

using namespace slamrs;

struct slamrs_gpu_handle {
    slamrs_gpu_config cfg{};
    int device = 0;
    int num_sms = 148;
    cudaStream_t stream = nullptr;
    cudaStream_t side_stream = nullptr;          // the planner runs here, next to the ray update
    cudaEvent_t ev_indices = nullptr, ev_plan = nullptr, ev_sort = nullptr;
    float2* d_valid_list = nullptr;     // (angle, distance) of the scan's valid beams (65,536 entries), filled by k_motion
    uint32_t* d_n_valid = nullptr;
    uint16_t* d_order = nullptr;   // beam order of the current scan for the ray kernel (SORT_MAX_BEAMS entries)
    bool order_valid = false, order_pending = false;

    uint32_t n_total = 0, n_local = 0, rank = 0, world = 1, first = 0;
    uint32_t n_cells = 0;        // grid_w * grid_h
    size_t cells_per_grid = 0;   // n_cells rounded up to 32 cells (128 B) so every slot is 128 B aligned
    uint32_t n_slots = 0, n_spare = 0;
    MapGeom geom{};

    // one allocation, mapped whole by the peers:
    // [SlotMeta x 2*n_local | ParticleResult x n_total | barrier flags | grid slots]
    void* d_pool = nullptr;
    size_t pool_header = 0;      // bytes in front of the first grid slot
    size_t off_results = 0, off_flags = 0, off_bands = 0, off_counters = 0;
    uint32_t* d_bands = nullptr;                 // band extents, n_bands entries per slot (inside the pool header)
    uint32_t n_bands = 0;
    uint32_t** d_peer_bands = nullptr;           // device array [world]
    unsigned long long* d_flags = nullptr;       // PEER_MAX_WORLD epochs, written by the peers
    ParticleResult** d_peer_results = nullptr;   // device array [world]
    std::vector<StepCounters*> peer_counters;    // host array [world]: every rank's step counters (inside its pool)
    unsigned long long** d_peer_flags = nullptr; // device array [world]
    unsigned long long barrier_epoch = 0;
    unsigned long long barrier_timeout_ns = 60000000000ull;   // SLAMRS_BARRIER_TIMEOUT_MS overrides
    bool p2p_exchange = false;   // fused peer stores + flag barriers instead of NCCL collectives
    SlotMeta* d_meta = nullptr;  // = d_pool
    uint32_t* d_cells = nullptr; // = d_pool + pool_header
    bool boxed_copy = false;     // extent-limited copies (needs rows that are multiples of 32 bytes)
    bool defer = false;          // clones share their source's cells until written (PlanArgs::alias_of)
    int32_t* d_alias = nullptr;  // n_slots
    CopyItem* d_mat_items = nullptr;     // n_local: shared grids made private before the ray update
    uint32_t* d_mat_leaders = nullptr;   // n_local
    uint32_t* d_mat_roots = nullptr;     // n_local scratch
    int32_t* d_slot[2] = {nullptr, nullptr};
    float* d_pose[2] = {nullptr, nullptr};
    int cur = 0;
    ParticleResult* d_results_base = nullptr;   // 2 x n_total records inside the pool header
    ParticleResult* d_results = nullptr;        // the generation of the last issued step
    double* d_wnorm = nullptr;
    double* d_cum = nullptr;
    double* d_fold = nullptr;    // scratch of k_weights' exact left fold
    double* d_carry = nullptr;   // adaptive resampling: weights carried over a step that did not resample (n_total)
    uint32_t* d_idx = nullptr;
    float* d_angle = nullptr;
    float* d_dist = nullptr;
    uint8_t* d_valid = nullptr;
    uint32_t beam_cap = 0, n_beams = 0;
    // host scans travel in ONE copy: d_angle | d_dist | d_valid are pieces of one allocation (d_angle is its base),
    // filled from a page-locked staging buffer of the same layout
    unsigned char* h_scan_stage = nullptr;
    cudaEvent_t ev_scan_uploaded = nullptr;
    bool scan_upload_pending = false;
    int radius_cells = 1;
    double* d_z = nullptr;
    double* d_u = nullptr;
    int32_t *d_keep = nullptr, *d_need = nullptr, *d_free = nullptr, *d_spare = nullptr;
    CopyItem* d_copies = nullptr;
    uint32_t* d_leaders = nullptr;
    void* d_jobs = nullptr;      // CopyJob scratch of the extent-limited copy
    uint32_t* d_alive = nullptr;
    RayItem* d_ray_items = nullptr;      // work list of the fused ray update (n_local)
    uint32_t* d_readers = nullptr;       // per slot: clones that read it in this step | per slot: clones that have (2 x n_slots)
    uint32_t* d_ray_spill = nullptr;     // scratch of the fused ray update
    void* d_ray_xchg = nullptr;          // per surviving particle: lower half -> upper half exchange record
    StepCounters* d_counters = nullptr;
    StepCounters* h_counters = nullptr;  // pinned
    double* d_export = nullptr;
    // pipelined map read-out (slamrs_gpu_map_probability_async): two export buffers, filled on the step's stream and
    // copied to the host on a stream of their own, so the copy overlaps the next step
    double* d_export_async[2] = {nullptr, nullptr};
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t ev_exported[2] = {nullptr, nullptr}, ev_copied[2] = {nullptr, nullptr};
    bool async_pending[2] = {false, false};
    int async_next = 0;
    double* d_term_table = nullptr;   // per-beam likelihood factor by hit-counter pair
    int* d_barrier = nullptr;

    Comm* comm = nullptr;
    uint32_t** d_peer_cells = nullptr;         // device array [world]
    SlotMeta** d_peer_meta = nullptr;          // device array [world]
    std::vector<void*> ipc_opened;             // peer mappings to close
    std::vector<uint32_t*> host_peer_cells;    // host copies of d_peer_cells / d_peer_meta
    std::vector<SlotMeta*> host_peer_meta;
    StepRecord* d_history = nullptr;
    bool scan_external = false;
    const float* ext_angle = nullptr;
    const float* ext_dist = nullptr;
    const uint8_t* ext_valid = nullptr;
    // profiling: per step SLAMRS_PHASE_COUNT+1 boundary events
    bool profiling = false;
    std::vector<cudaEvent_t> prof_events;   // [PROF_RING][SLAMRS_PHASE_COUNT + 1]
    uint32_t prof_recorded = 0;
    double prof_ms[SLAMRS_PHASE_COUNT] = {0, 0, 0, 0, 0, 0, 0};
    uint64_t prof_steps = 0;
    uint64_t step = 0;
    bool counters_fresh = false;   // h_counters mirrors d_counters (no step issued since the last fetch)
    bool mirror_by_step = false;   // the last issued step writes the mirror itself (its last kernel): a fetch only synchronises
    bool mirror_wanted = false;    // set by slamrs_gpu_update around its step: the caller synchronises right behind it
    bool est_box_stale = false;    // set_cells changed a grid after the step recorded the estimate's extent
    uint64_t launches = 0;
    uint64_t window_cells = 0;
    std::string last_error;
    // localiser mode (slamrs_gpu_create_localizer): one shared map as a per-cell term table, no grids
    bool localizer = false;
    double* d_loc_terms = nullptr;   // n_cells
    double loc_outside = 0.0;        // term of an endpoint off the grid
    // scan-matching pose refinement (slamrs_gpu_set_scan_match)
    bool match_on = false;
    ScanMatchParams match{};
    uint2* d_match_stats = nullptr;  // n_local x {moves, poses scored} of the last step that ran the matcher
    bool match_last_step = false;    // the last issued step ran it
    uint32_t match_last_max_moves = 0;
};

namespace {

thread_local std::string g_create_error;

int fail(slamrs_gpu_handle* h, int code, const std::string& msg) {
    if (h) h->last_error = msg;
    else g_create_error = msg;
    return code;
}

#define CU_TRY(h, expr)                                                                               \
    do {                                                                                              \
        cudaError_t _e = (expr);                                                                      \
        if (_e != cudaSuccess) {                                                                      \
            const int _code = (_e == cudaErrorMemoryAllocation) ? SLAMRS_E_OUT_OF_MEMORY : SLAMRS_E_CUDA; \
            return fail(h, _code, std::string(#expr) + ": " + cudaGetErrorString(_e));                \
        }                                                                                             \
    } while (0)

// Odometry::new, slamrs/common/src/robot.rs:132-150
OdomModel odometry_new(float dl, float dr, float wheel) {
    OdomModel o;
    const double delta_center = (double)((dl + dr) / 2.0f);
    const double delta_theta = (double)((dr - dl) / wheel);
    o.mean_c = delta_center;
    o.std_c = (0.01 + fabs(delta_center) * 0.05) / 2.0;
    const double rads_per_deg = 3.14159265358979323846264338327950288 / 180.0;  // f64::to_radians
    o.mean_t = delta_theta;
    o.std_t = 5.0 * rads_per_deg + 0.1 * fabs(delta_theta);
    return o;
}

struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int dev) {
        cudaGetDevice(&prev);
        if (prev != dev) cudaSetDevice(dev);
    }
    ~DeviceGuard() {
        int now = -1;
        cudaGetDevice(&now);
        if (prev >= 0 && now != prev) cudaSetDevice(prev);
    }
};

struct PeerInfo {  // exchanged between ranks at create
    cudaIpcMemHandle_t handle;
    uint64_t pid;
    uint64_t ptr;
    int32_t device;
    int32_t pad;
};

int setup_peers(slamrs_gpu_handle* h) {
    const uint32_t W = h->world;
    std::vector<PeerInfo> all(W);
    PeerInfo mine;
    memset(&mine, 0, sizeof(mine));
    CU_TRY(h, cudaIpcGetMemHandle(&mine.handle, h->d_pool));
    mine.pid = (uint64_t)getpid();
    mine.ptr = (uint64_t)(uintptr_t)h->d_pool;
    mine.device = h->device;
    PeerInfo* d_all = nullptr;
    CU_TRY(h, cudaMalloc(&d_all, sizeof(PeerInfo) * W));
    CU_TRY(h, cudaMemcpyAsync(d_all + h->rank, &mine, sizeof(mine), cudaMemcpyHostToDevice, h->stream));
    std::string err;
    if (comm_all_gather(h->comm, d_all + h->rank, d_all, sizeof(PeerInfo), h->stream, &err)) {
        cudaFree(d_all);
        return fail(h, SLAMRS_E_NCCL, err);
    }
    CU_TRY(h, cudaMemcpyAsync(all.data(), d_all, sizeof(PeerInfo) * W, cudaMemcpyDeviceToHost, h->stream));
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    cudaFree(d_all);

    std::vector<char*> peers(W, nullptr);   // pool base of every rank (same header size everywhere)
    for (uint32_t r = 0; r < W; ++r) {
        if (r == h->rank) { peers[r] = (char*)h->d_pool; continue; }
        if (all[r].pid == mine.pid) {
            // same process: plain peer access to the other device's allocation
            int can = 0;
            CU_TRY(h, cudaDeviceCanAccessPeer(&can, h->device, all[r].device));
            if (!can) return fail(h, SLAMRS_E_CUDA, "peer access between GPUs not available");
            cudaError_t e = cudaDeviceEnablePeerAccess(all[r].device, 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled)
                return fail(h, SLAMRS_E_CUDA, std::string("cudaDeviceEnablePeerAccess: ") + cudaGetErrorString(e));
            cudaGetLastError();
            peers[r] = (char*)(uintptr_t)all[r].ptr;
        } else {
            void* p = nullptr;
            CU_TRY(h, cudaIpcOpenMemHandle(&p, all[r].handle, cudaIpcMemLazyEnablePeerAccess));
            h->ipc_opened.push_back(p);
            peers[r] = (char*)p;
        }
    }
    std::vector<uint32_t*> pcells(W);
    std::vector<SlotMeta*> pmeta(W);
    std::vector<ParticleResult*> pres(W);
    std::vector<unsigned long long*> pflags(W);
    std::vector<uint32_t*> pbands(W);
    for (uint32_t r = 0; r < W; ++r) {
        pmeta[r] = (SlotMeta*)peers[r];
        pcells[r] = (uint32_t*)(peers[r] + h->pool_header);
        pres[r] = (ParticleResult*)(peers[r] + h->off_results);
        pflags[r] = (unsigned long long*)(peers[r] + h->off_flags);
        pbands[r] = (uint32_t*)(peers[r] + h->off_bands);
        h->peer_counters[r] = (StepCounters*)(peers[r] + h->off_counters);
    }
    h->host_peer_cells = pcells;
    h->host_peer_meta = pmeta;
    CU_TRY(h, cudaMalloc(&h->d_peer_bands, sizeof(uint32_t*) * W));
    CU_TRY(h, cudaMemcpy(h->d_peer_bands, pbands.data(), sizeof(uint32_t*) * W, cudaMemcpyHostToDevice));
    CU_TRY(h, cudaMalloc(&h->d_peer_results, sizeof(ParticleResult*) * W));
    CU_TRY(h, cudaMemcpy(h->d_peer_results, pres.data(), sizeof(ParticleResult*) * W, cudaMemcpyHostToDevice));
    CU_TRY(h, cudaMalloc(&h->d_peer_flags, sizeof(unsigned long long*) * W));
    CU_TRY(h, cudaMemcpy(h->d_peer_flags, pflags.data(), sizeof(unsigned long long*) * W, cudaMemcpyHostToDevice));
    CU_TRY(h, cudaMalloc(&h->d_peer_cells, sizeof(uint32_t*) * W));
    CU_TRY(h, cudaMemcpy(h->d_peer_cells, pcells.data(), sizeof(uint32_t*) * W, cudaMemcpyHostToDevice));
    CU_TRY(h, cudaMalloc(&h->d_peer_meta, sizeof(SlotMeta*) * W));
    CU_TRY(h, cudaMemcpy(h->d_peer_meta, pmeta.data(), sizeof(SlotMeta*) * W, cudaMemcpyHostToDevice));
    return SLAMRS_OK;
}

void free_all(slamrs_gpu_handle* h) {
    if (!h) return;
    DeviceGuard g(h->device);
    if (h->side_stream) cudaStreamSynchronize(h->side_stream);
    if (h->stream) cudaStreamSynchronize(h->stream);
    if (h->comm && h->d_barrier && h->stream) {
        // Nobody may still be reading or writing this pool when it is freed: say goodbye and wait until
        // every peer has said it too (k_peer_barrier). A peer that is still stepping meets the goodbye at
        // its next barrier, fails that step and is destroyed by its owner, which releases this rank. The
        // wait is bounded by the barrier timeout (a dead peer process never answers); a handle that is
        // already poisoned publishes its goodbye and does not wait.
        if (h->p2p_exchange && h->d_peer_flags) {
            launch_peer_goodbye(h->stream, h->d_peer_flags, h->d_flags, h->rank, h->world, h->barrier_timeout_ns,
                                h->d_counters);
            cudaStreamSynchronize(h->stream);
        } else {
            std::string err;
            if (comm_barrier(h->comm, h->d_barrier, h->stream, &err) == 0) cudaStreamSynchronize(h->stream);
        }
    }
    for (void* p : h->ipc_opened) cudaIpcCloseMemHandle(p);
    h->ipc_opened.clear();
    comm_destroy(h->comm);
    h->comm = nullptr;
    cudaFree(h->d_pool);
    cudaFree(h->d_slot[0]); cudaFree(h->d_slot[1]);
    cudaFree(h->d_pose[0]); cudaFree(h->d_pose[1]);
    cudaFree(h->d_term_table); cudaFree(h->d_loc_terms);
    cudaFree(h->d_wnorm); cudaFree(h->d_cum); cudaFree(h->d_idx); cudaFree(h->d_fold); cudaFree(h->d_carry);
    cudaFree(h->d_angle);   // (d_dist and d_valid live in the same allocation)
    if (h->h_scan_stage) cudaFreeHost(h->h_scan_stage);
    if (h->ev_scan_uploaded) cudaEventDestroy(h->ev_scan_uploaded);
    cudaFree(h->d_z); cudaFree(h->d_u);
    cudaFree(h->d_keep); cudaFree(h->d_need); cudaFree(h->d_free); cudaFree(h->d_spare);
    cudaFree(h->d_copies); cudaFree(h->d_leaders); cudaFree(h->d_alive); cudaFree(h->d_jobs);
    cudaFree(h->d_ray_items); cudaFree(h->d_readers); cudaFree(h->d_ray_spill); cudaFree(h->d_ray_xchg);
    cudaFree(h->d_alias); cudaFree(h->d_mat_items); cudaFree(h->d_mat_leaders); cudaFree(h->d_mat_roots);
    cudaFree(h->d_export); cudaFree(h->d_barrier); cudaFree(h->d_peer_cells); cudaFree(h->d_peer_meta);
    cudaFree(h->d_peer_results); cudaFree(h->d_peer_flags); cudaFree(h->d_peer_bands);
    cudaFree(h->d_history);
    for (cudaEvent_t e : h->prof_events) cudaEventDestroy(e);
    h->prof_events.clear();
    if (h->h_counters) cudaFreeHost(h->h_counters);
    if (h->ev_indices) cudaEventDestroy(h->ev_indices);
    if (h->ev_plan) cudaEventDestroy(h->ev_plan);
    if (h->ev_sort) cudaEventDestroy(h->ev_sort);
    cudaFree(h->d_order); cudaFree(h->d_valid_list); cudaFree(h->d_n_valid);
    cudaFree(h->d_match_stats);
    if (h->copy_stream) { cudaStreamSynchronize(h->copy_stream); cudaStreamDestroy(h->copy_stream); }
    for (int k = 0; k < 2; ++k) {
        cudaFree(h->d_export_async[k]);
        if (h->ev_exported[k]) cudaEventDestroy(h->ev_exported[k]);
        if (h->ev_copied[k]) cudaEventDestroy(h->ev_copied[k]);
    }
    if (h->side_stream) cudaStreamDestroy(h->side_stream);
    if (h->stream) cudaStreamDestroy(h->stream);
    cudaGetLastError();
    delete h;
}

constexpr const char* NO_GRIDS = "a localizer has no particle grids";

int ensure_beam_capacity(slamrs_gpu_handle* h, uint32_t n) {
    if (n <= h->beam_cap) return SLAMRS_OK;
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    cudaFree(h->d_angle);
    if (h->h_scan_stage) cudaFreeHost(h->h_scan_stage);
    h->d_angle = h->d_dist = nullptr; h->d_valid = nullptr; h->h_scan_stage = nullptr; h->beam_cap = 0;
    h->scan_upload_pending = false;
    const uint32_t cap = (n + 255u) & ~255u;
    unsigned char* base = nullptr;
    CU_TRY(h, cudaMalloc(&base, 9u * (size_t)cap));
    h->d_angle = reinterpret_cast<float*>(base);
    h->d_dist = reinterpret_cast<float*>(base + 4u * (size_t)cap);
    h->d_valid = base + 8u * (size_t)cap;
    CU_TRY(h, cudaMallocHost(&h->h_scan_stage, 9u * (size_t)cap));
    if (!h->ev_scan_uploaded) CU_TRY(h, cudaEventCreateWithFlags(&h->ev_scan_uploaded, cudaEventDisableTiming));
    h->beam_cap = cap;
    return SLAMRS_OK;
}

constexpr uint32_t PROF_RING = 64;
constexpr uint32_t PROF_MARKS = SLAMRS_PHASE_COUNT + 1;

int prof_flush(slamrs_gpu_handle* h) {
    if (h->prof_recorded == 0) return SLAMRS_OK;
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    for (uint32_t r = 0; r < h->prof_recorded; ++r) {
        for (int p = 0; p < SLAMRS_PHASE_COUNT; ++p) {
            float ms = 0.f;
            CU_TRY(h, cudaEventElapsedTime(&ms, h->prof_events[r * PROF_MARKS + p], h->prof_events[r * PROF_MARKS + p + 1]));
            h->prof_ms[p] += ms;
        }
    }
    h->prof_steps += h->prof_recorded;
    h->prof_recorded = 0;
    return SLAMRS_OK;
}

// records boundary mark `m` of the current step when profiling is on
#define PROF_MARK(h, m)                                                                                   \
    do {                                                                                                  \
        if ((h)->profiling) CU_TRY(h, cudaEventRecord((h)->prof_events[(h)->prof_recorded * PROF_MARKS + (m)], (h)->stream)); \
    } while (0)

// the copies k_materialize_list has listed: shared grids get their own cells (extent copies)
int materialize_copies(slamrs_gpu_handle* h, bool grouped) {
    launch_copy_boxed(h->stream, h->d_mat_items, grouped ? h->d_mat_leaders : nullptr, &h->d_counters->n_mat,
                      &h->d_counters->n_mat_leaders, h->n_local, h->d_jobs, h->geom, h->d_counters, h->num_sms, !grouped);
    launch_commit_boxes(h->stream, h->d_mat_items, &h->d_counters->n_mat, h->n_local, h->geom, true, h->d_counters, nullptr);
    h->launches += 3;
    return SLAMRS_OK;
}
// every local grid private again (before a grid is overwritten from the host: its clones must not follow)
int unshare_all(slamrs_gpu_handle* h) {
    if (!h->defer) return SLAMRS_OK;
    launch_materialize_list(h->stream, nullptr, h->n_total, h->first, h->n_local, h->d_slot[h->cur], h->d_alias, h->d_cells,
                            h->cells_per_grid, h->d_meta, h->d_bands, h->n_bands, h->d_mat_items, h->d_mat_leaders,
                            h->d_mat_roots, h->d_counters);
    h->launches++;
    int rc = materialize_copies(h, true);
    if (rc) return rc;
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    h->counters_fresh = false;
    h->mirror_by_step = false;
    return SLAMRS_OK;
}

// stream-ordered barrier across ranks inside a step: peer flags by default, NCCL on request
int step_barrier(slamrs_gpu_handle* h) {
    if (h->p2p_exchange) {
        launch_peer_barrier(h->stream, h->d_peer_flags, h->d_flags, h->rank, h->world, ++h->barrier_epoch,
                            h->barrier_timeout_ns, h->d_counters);
        h->launches++;
        return SLAMRS_OK;
    }
    std::string err;
    if (comm_barrier(h->comm, h->d_barrier, h->stream, &err)) return fail(h, SLAMRS_E_NCCL, err);
    return SLAMRS_OK;
}

// Host copy of the device counters. They only change when a step is issued, so one fetch (with its
// stream synchronisation) serves every read-out that follows the same step.
int fetch_counters(slamrs_gpu_handle* h) {
    if (h->counters_fresh) return SLAMRS_OK;
    if (!h->mirror_by_step) {
        launch_publish_counters(h->stream, h->d_counters, h->h_counters);   // (not a memcpy: see k_publish_counters)
        h->launches++;
    }
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    CU_TRY(h, cudaGetLastError());
    h->counters_fresh = true;
    return SLAMRS_OK;
}

// One localisation step (localiser mode): motion + likelihood against the term table, then the SLAM step's own
// weights and resampling kernels without a survivor list -- three launches, chained by programmatic dependent launch.
int loc_step_async(slamrs_gpu_handle* h, const OdomModel& od, bool caller) {
    cudaStream_t s = h->stream;
    if (h->profiling && h->prof_recorded == PROF_RING) {
        int prc = prof_flush(h);
        if (prc) return prc;
    }
    const int cur = h->cur, nxt = cur ^ 1;
    const ScanDevice scan = h->scan_external ? ScanDevice{h->ext_angle, h->ext_dist, h->ext_valid, h->n_beams, nullptr}
                                             : ScanDevice{h->d_angle, h->d_dist, h->d_valid, h->n_beams, nullptr};
    PROF_MARK(h, 0);
    launch_loc_step(s, h->geom, od, scan, h->d_pose[cur], h->d_results, h->n_total, caller ? h->d_z : nullptr, h->cfg.seed,
                    h->step, h->d_loc_terms, h->loc_outside, h->d_carry, h->d_counters);
    PROF_MARK(h, 1);
    PROF_MARK(h, 2);
    launch_weights(s, h->d_results, h->n_total, h->d_wnorm, h->d_cum, h->d_fold, (double)h->cfg.resample_threshold, h->d_counters);
    launch_resample_indices(s, h->d_results, h->d_cum, h->n_total, caller ? h->d_u : nullptr, h->cfg.seed, h->step, h->d_idx,
                            h->d_pose[nxt], 0, h->n_total, false, nullptr,
                            RayLists{nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, 0u, 0u}, h->d_wnorm, h->d_carry,
                            h->d_counters);
    h->launches += 3;
    for (uint32_t m = 3; m < PROF_MARKS; ++m) PROF_MARK(h, m);
    if (h->profiling) h->prof_recorded++;
    CU_TRY(h, cudaGetLastError());
    h->cur = nxt;
    h->step++;
    h->counters_fresh = false;
    h->mirror_by_step = false;
    return SLAMRS_OK;
}

}  // namespace

namespace {
template <typename T>
struct DevBuf {
    T* p = nullptr;
    cudaError_t alloc(size_t n) { return cudaMalloc(&p, sizeof(T) * (n ? n : 1)); }
    ~DevBuf() { cudaFree(p); }
};
int debug_device(int device) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) { cudaGetLastError(); return SLAMRS_E_NO_DEVICE; }
    if (device >= n) return SLAMRS_E_INVALID_ARG;
    return SLAMRS_OK;
}
#define DBG_CU(expr)                                                                     \
    do {                                                                                 \
        cudaError_t _e = (expr);                                                         \
        if (_e != cudaSuccess) return fail(nullptr, SLAMRS_E_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e)); \
    } while (0)
}  // namespace

extern "C" {

int slamrs_gpu_grid_cells(float extent, float resolution, uint32_t* out_cells) {
    if (!out_cells) return SLAMRS_E_INVALID_ARG;
    const float c = ceilf(extent / resolution);  // map.rs:28-31, f32 division then ceil, `as usize` saturates
    if (!(c == c) || c <= 0.0f) { *out_cells = 0; return SLAMRS_OK; }
    if (c >= 4294967296.0f) return SLAMRS_E_INVALID_ARG;
    *out_cells = (uint32_t)c;
    return SLAMRS_OK;
}

int slamrs_gpu_nccl_unique_id(uint8_t out[SLAMRS_NCCL_ID_BYTES]) {
    if (!out) return SLAMRS_E_INVALID_ARG;
    std::string err;
    if (comm_unique_id(out, &err)) return fail(nullptr, SLAMRS_E_NCCL, err);
    return SLAMRS_OK;
}

int slamrs_gpu_create(const slamrs_gpu_config* cfg, slamrs_gpu_handle** out) {
    if (!cfg || !out) return fail(nullptr, SLAMRS_E_INVALID_ARG, "null config or output pointer");
    *out = nullptr;
    if (cfg->struct_size != sizeof(slamrs_gpu_config) || cfg->abi_version != SLAMRS_GPU_ABI_VERSION)
        return fail(nullptr, SLAMRS_E_INVALID_ARG, "slamrs_gpu_config size/ABI version mismatch");
    if (cfg->n_particles == 0)  // ParticleFilter::new asserts, particle.rs:16
        return fail(nullptr, SLAMRS_E_INVALID_ARG, "Must have at least one particle");
    if (cfg->world_size > PEER_MAX_WORLD) return fail(nullptr, SLAMRS_E_INVALID_ARG, "world_size above 64");
    // the fused exchange stores one record per lane of the likelihood warp: at most 32 peers
    if (cfg->world_size > 32u && (cfg->flags & SLAMRS_FLAG_NCCL_EXCHANGE) == 0)
        return fail(nullptr, SLAMRS_E_INVALID_ARG, "world_size above 32 needs SLAMRS_FLAG_NCCL_EXCHANGE (the peer-store exchange serves 32 GPUs)");
    if (cfg->world_size == 0 || cfg->rank >= cfg->world_size || cfg->n_particles % cfg->world_size != 0)
        return fail(nullptr, SLAMRS_E_INVALID_ARG, "bad rank/world_size or n_particles not divisible by world_size");
    if (cfg->n_particles > 0x7fffffffull) return fail(nullptr, SLAMRS_E_INVALID_ARG, "too many particles");
    if (cfg->grid_w == 0 || cfg->grid_w != cfg->grid_h)
        return fail(nullptr, SLAMRS_E_INVALID_ARG,
                    "grid must be square and non-empty (the reference index row*size.y+column aliases otherwise)");
    if ((uint64_t)cfg->grid_w * cfg->grid_h > 0x7fffffffull) return fail(nullptr, SLAMRS_E_INVALID_ARG, "grid too large");
    if (!(cfg->resolution > 0.0f)) return fail(nullptr, SLAMRS_E_INVALID_ARG, "resolution must be positive");
    if (cfg->rng_mode > SLAMRS_RNG_CALLER) return fail(nullptr, SLAMRS_E_INVALID_ARG, "unknown rng_mode");
    if (!(cfg->resample_threshold >= 0.0f && cfg->resample_threshold <= 1.0f))
        return fail(nullptr, SLAMRS_E_INVALID_ARG, "resample_threshold must be 0 (always resample) or in (0, 1]");
    if (cfg->slot_cells != 0 && (cfg->slot_cells < 256u || (cfg->slot_cells & (cfg->slot_cells - 1u)) != 0u))
        return fail(nullptr, SLAMRS_E_INVALID_ARG, "slot_cells must be 0 (whole grid) or a power of two >= 256");

    int n_dev = 0;
    if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev == 0) {
        cudaGetLastError();
        return fail(nullptr, SLAMRS_E_NO_DEVICE, "no CUDA device visible; this library has no CPU fallback");
    }
    int device = cfg->device;
    if (device < 0) cudaGetDevice(&device);
    if (device >= n_dev) return fail(nullptr, SLAMRS_E_INVALID_ARG, "device ordinal out of range");

    slamrs_gpu_handle* h = new (std::nothrow) slamrs_gpu_handle();
    if (!h) return fail(nullptr, SLAMRS_E_OUT_OF_MEMORY, "host allocation failed");
    h->cfg = *cfg;
    h->device = device;
    h->world = cfg->world_size;
    h->rank = cfg->rank;
    h->n_total = (uint32_t)cfg->n_particles;
    h->n_local = h->n_total / h->world;
    h->first = h->rank * h->n_local;
    h->n_cells = cfg->grid_w * cfg->grid_h;
    h->geom = make_map_geom(cfg->pos_x, cfg->pos_y, cfg->resolution, cfg->grid_w, cfg->grid_h, cfg->slot_cells);
    // a slot holds pw x ph cells: the whole grid, or (windowed slots) a power-of-two torus of it
    h->cells_per_grid = ((size_t)h->geom.pw * h->geom.ph + 31u) & ~(size_t)31u;

#define CREATE_TRY(expr)                                  \
    do {                                                  \
        int _rc = (expr);                                 \
        if (_rc != SLAMRS_OK) {                           \
            g_create_error = h->last_error;               \
            free_all(h);                                  \
            return _rc;                                   \
        }                                                 \
    } while (0)
#define CREATE_CU(expr)                                                                                   \
    do {                                                                                                  \
        cudaError_t _e = (expr);                                                                          \
        if (_e != cudaSuccess) {                                                                          \
            const int _code = (_e == cudaErrorMemoryAllocation) ? SLAMRS_E_OUT_OF_MEMORY : SLAMRS_E_CUDA; \
            g_create_error = std::string(#expr) + ": " + cudaGetErrorString(_e);                          \
            cudaGetLastError();                                                                           \
            free_all(h);                                                                                  \
            return _code;                                                                                 \
        }                                                                                                 \
    } while (0)

    DeviceGuard guard(device);
    cudaDeviceProp prop;
    CREATE_CU(cudaGetDeviceProperties(&prop, device));
    h->num_sms = prop.multiProcessorCount;
    if (prop.major < 10) {
        g_create_error = "this library is built for sm_100a (B200) only";
        free_all(h);
        return SLAMRS_E_NO_DEVICE;
    }
    CREATE_CU(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
    CREATE_CU(cudaStreamCreateWithFlags(&h->side_stream, cudaStreamNonBlocking));
    CREATE_CU(cudaEventCreateWithFlags(&h->ev_indices, cudaEventDisableTiming));
    CREATE_CU(cudaEventCreateWithFlags(&h->ev_plan, cudaEventDisableTiming));
    CREATE_CU(cudaEventCreateWithFlags(&h->ev_sort, cudaEventDisableTiming));
    CREATE_CU(cudaMalloc(&h->d_order, sizeof(uint16_t) * SORT_MAX_BEAMS));
    CREATE_CU(cudaMalloc(&h->d_valid_list, sizeof(float2) * 65536));
    CREATE_CU(cudaMalloc(&h->d_n_valid, sizeof(uint32_t)));
    CREATE_CU(configure_kernels());

    // spare slots: staging room for grids that migrate between GPUs at resampling
    const size_t grid_bytes = h->cells_per_grid * sizeof(uint32_t);
    if (h->world > 1) {
        uint32_t spare = cfg->spare_slots;
        if (spare == 0) {
            size_t free_b = 0, total_b = 0;
            CREATE_CU(cudaMemGetInfo(&free_b, &total_b));
            const size_t reserve = (size_t)2 << 30;  // leave room for NCCL buffers and small arrays
            const size_t live = (size_t)h->n_local * grid_bytes;
            size_t room = free_b > live + reserve ? (free_b - live - reserve) / grid_bytes : 0;
            spare = (uint32_t)(room < h->n_local ? room : h->n_local);
        }
        h->n_spare = spare;
    }
    h->n_slots = h->n_local + h->n_spare;

    // the header holds one SlotMeta per possible slot; its size depends on n_local only, so every
    // rank can locate a peer's slots and extents from the peer's pool base alone
    h->off_results = (sizeof(SlotMeta) * 2 * (size_t)h->n_local + 255) & ~(size_t)255;
    // two generations of the population array (step parity): a peer that is one step ahead stores
    // its next records while this rank's host may still be reading the last step's
    h->off_flags = (h->off_results + 2 * sizeof(ParticleResult) * (size_t)h->n_total + 255) & ~(size_t)255;
    h->n_bands = bands_per_slot(h->geom);
    h->off_bands = (h->off_flags + sizeof(unsigned long long) * 2 * PEER_MAX_WORLD + 255) & ~(size_t)255;   // epochs | goodbyes
    // the step counters live in the header too: a peer that reads out the published map finds the estimate's slot there
    h->off_counters = (h->off_bands + sizeof(uint32_t) * 2 * (size_t)h->n_local * h->n_bands + 255) & ~(size_t)255;
    h->pool_header = (h->off_counters + sizeof(StepCounters) + 4095) & ~(size_t)4095;
    CREATE_CU(cudaMalloc(&h->d_pool, h->pool_header + (size_t)h->n_slots * grid_bytes));
    h->d_meta = (SlotMeta*)h->d_pool;
    h->d_cells = (uint32_t*)((char*)h->d_pool + h->pool_header);
    h->d_results_base = (ParticleResult*)((char*)h->d_pool + h->off_results);   // zeroed with the pool
    h->d_results = h->d_results_base;
    h->d_flags = (unsigned long long*)((char*)h->d_pool + h->off_flags);
    h->d_bands = (uint32_t*)((char*)h->d_pool + h->off_bands);
    h->d_counters = (StepCounters*)((char*)h->d_pool + h->off_counters);
    h->peer_counters.assign(h->world, nullptr);
    h->peer_counters[h->rank] = h->d_counters;
    h->p2p_exchange = h->world > 1 && (cfg->flags & SLAMRS_FLAG_NCCL_EXCHANGE) == 0;
    CREATE_CU(cudaMemsetAsync(h->d_pool, 0, h->pool_header + (size_t)h->n_slots * grid_bytes, h->stream));  // ln(0.5/0.5) = 0
    h->boxed_copy = (cfg->flags & SLAMRS_FLAG_FULL_GRID_COPY) == 0 && cfg->grid_w % 8u == 0u && h->geom.pw % 8u == 0u;
    h->defer = h->boxed_copy && (cfg->flags & SLAMRS_FLAG_EAGER_COPY) == 0;
    for (int i = 0; i < 2; ++i) {
        CREATE_CU(cudaMalloc(&h->d_slot[i], sizeof(int32_t) * h->n_local));
        CREATE_CU(cudaMalloc(&h->d_pose[i], sizeof(float) * 3 * h->n_local));
        CREATE_CU(cudaMemsetAsync(h->d_pose[i], 0, sizeof(float) * 3 * h->n_local, h->stream));  // Pose::default()
    }
    CREATE_CU(cudaMalloc(&h->d_wnorm, sizeof(double) * h->n_total));
    CREATE_CU(cudaMalloc(&h->d_cum, sizeof(double) * h->n_total));
    CREATE_CU(cudaMalloc(&h->d_idx, sizeof(uint32_t) * h->n_total));
    CREATE_CU(cudaMalloc(&h->d_fold, sizeof(double) * weights_scratch_doubles()));
    if (cfg->resample_threshold > 0.0f) CREATE_CU(cudaMalloc(&h->d_carry, sizeof(double) * h->n_total));
    CREATE_CU(cudaMemsetAsync(h->d_wnorm, 0, sizeof(double) * h->n_total, h->stream));
    CREATE_CU(cudaMemsetAsync(h->d_idx, 0, sizeof(uint32_t) * h->n_total, h->stream));
    if (cfg->rng_mode == SLAMRS_RNG_CALLER) {
        CREATE_CU(cudaMalloc(&h->d_z, sizeof(double) * 2 * h->n_total));
        CREATE_CU(cudaMalloc(&h->d_u, sizeof(double)));
    }
    CREATE_CU(cudaMalloc(&h->d_keep, sizeof(int32_t) * h->n_local));
    CREATE_CU(cudaMalloc(&h->d_need, sizeof(int32_t) * h->n_local));
    CREATE_CU(cudaMalloc(&h->d_free, sizeof(int32_t) * ((size_t)h->n_local + h->n_spare + 1)));
    CREATE_CU(cudaMalloc(&h->d_spare, sizeof(int32_t) * ((size_t)h->n_spare + 1)));
    CREATE_CU(cudaMalloc(&h->d_copies, sizeof(CopyItem) * h->n_local));
    CREATE_CU(cudaMalloc(&h->d_leaders, sizeof(uint32_t) * h->n_local));
    CREATE_CU(cudaMalloc(&h->d_jobs, copy_job_bytes() * h->n_local));
    CREATE_CU(cudaMalloc(&h->d_alias, sizeof(int32_t) * h->n_slots));
    CREATE_CU(cudaMalloc(&h->d_mat_items, sizeof(CopyItem) * h->n_local));
    CREATE_CU(cudaMalloc(&h->d_mat_leaders, sizeof(uint32_t) * h->n_local));
    CREATE_CU(cudaMalloc(&h->d_mat_roots, sizeof(uint32_t) * h->n_local));
    CREATE_CU(cudaMalloc(&h->d_alive, sizeof(uint32_t) * h->n_local));
    CREATE_CU(cudaMalloc(&h->d_ray_items, sizeof(RayItem) * 2 * (size_t)h->n_local));   // clones | owners
    CREATE_CU(cudaMalloc(&h->d_readers, sizeof(uint32_t) * (2 * (size_t)h->n_slots + 2 * (size_t)h->n_local)));   // readers | done | xflag | xdone
    CREATE_CU(cudaMalloc(&h->d_ray_xchg, ray_half_xchg_bytes() * h->n_local));
    CREATE_CU(cudaMalloc(&h->d_ray_spill, sizeof(uint32_t) * ray_spill_scratch_words(h->num_sms)));
    CREATE_CU(cudaMallocHost(&h->h_counters, sizeof(StepCounters)));
    memset(h->h_counters, 0, sizeof(StepCounters));
    CREATE_CU(cudaMalloc(&h->d_export, sizeof(double) * h->n_cells));
    // the pipelined read-out's buffers exist from the start: no allocation (an implicit device synchronisation) later
    CREATE_CU(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
    for (int k = 0; k < 2; ++k) {
        CREATE_CU(cudaMalloc(&h->d_export_async[k], sizeof(double) * h->n_cells));
        CREATE_CU(cudaEventCreateWithFlags(&h->ev_exported[k], cudaEventDisableTiming));
        CREATE_CU(cudaEventCreateWithFlags(&h->ev_copied[k], cudaEventDisableTiming));
    }
    CREATE_CU(cudaMalloc(&h->d_term_table, sizeof(double) * LK_TABLE_NF * LK_TABLE_NO));
    launch_fill_term_table(h->stream, h->d_term_table);
    h->launches++;
    CREATE_CU(cudaMalloc(&h->d_history, sizeof(StepRecord) * STEP_HISTORY));
    CREATE_CU(cudaMemsetAsync(h->d_history, 0xff, sizeof(StepRecord) * STEP_HISTORY, h->stream));
    CREATE_CU(cudaMalloc(&h->d_barrier, sizeof(int)));
    CREATE_CU(cudaMemsetAsync(h->d_barrier, 0, sizeof(int), h->stream));
    launch_init_slots(h->stream, h->d_slot[0], h->n_local, h->d_spare, h->n_spare, h->d_counters, h->rank, h->d_meta, h->d_alias);
    h->launches++;
    CREATE_CU(cudaGetLastError());

    if (h->world > 1) {
        std::string err;
        h->comm = comm_create(cfg->nccl_id, (int)h->rank, (int)h->world, &err);
        if (!h->comm) {
            g_create_error = err;
            free_all(h);
            return SLAMRS_E_NCCL;
        }
        CREATE_TRY(setup_peers(h));
        if (const char* ev = getenv("SLAMRS_BARRIER_TIMEOUT_MS")) {
            const long long ms = atoll(ev);
            if (ms > 0) h->barrier_timeout_ns = (unsigned long long)ms * 1000000ull;
        }
        // leave create together: mapping the peers' pools takes a rank-dependent time
        if (comm_barrier(h->comm, h->d_barrier, h->stream, &err)) {
            g_create_error = err;
            free_all(h);
            return SLAMRS_E_NCCL;
        }
    }
    CREATE_CU(cudaStreamSynchronize(h->stream));
    h->h_counters->est_slot = h->rank == 0 ? 0 : -1;
    h->h_counters->n_spare = h->n_spare;
#undef CREATE_TRY
#undef CREATE_CU
    *out = h;
    return SLAMRS_OK;
}

int slamrs_gpu_create_localizer(const slamrs_gpu_config* cfg, const slamrs_gpu_sensor_model* model,
                                const double* map_probability, slamrs_gpu_handle** out) {
    if (!out) return fail(nullptr, SLAMRS_E_INVALID_ARG, "null output pointer");
    *out = nullptr;
    if (!cfg) return fail(nullptr, SLAMRS_E_INVALID_ARG, "null config");
    if (!model) return fail(nullptr, SLAMRS_E_INVALID_ARG, "null sensor model");
    if (!map_probability) return fail(nullptr, SLAMRS_E_INVALID_ARG, "null map_probability");
    if (cfg->struct_size != sizeof(slamrs_gpu_config) || cfg->abi_version != SLAMRS_GPU_ABI_VERSION)
        return fail(nullptr, SLAMRS_E_INVALID_ARG, "slamrs_gpu_config size/ABI version mismatch");
    if (model->struct_size != sizeof(slamrs_gpu_sensor_model))
        return fail(nullptr, SLAMRS_E_INVALID_ARG, "slamrs_gpu_sensor_model struct_size mismatch");
    if (cfg->n_particles == 0) return fail(nullptr, SLAMRS_E_INVALID_ARG, "Must have at least one particle");
    if (cfg->n_particles > 0x7fffffffull) return fail(nullptr, SLAMRS_E_INVALID_ARG, "too many particles");
    if (cfg->world_size != 1 || cfg->rank != 0)
        return fail(nullptr, SLAMRS_E_INVALID_ARG, "world_size must be 1 and rank 0: a localizer runs on one GPU");
    if (cfg->flags != 0) return fail(nullptr, SLAMRS_E_INVALID_ARG, "flags must be 0 for a localizer");
    if (cfg->slot_cells != 0) return fail(nullptr, SLAMRS_E_INVALID_ARG, "slot_cells must be 0 for a localizer");
    if (cfg->spare_slots != 0) return fail(nullptr, SLAMRS_E_INVALID_ARG, "spare_slots must be 0 for a localizer");
    if (cfg->grid_w == 0 || cfg->grid_w != cfg->grid_h)
        return fail(nullptr, SLAMRS_E_INVALID_ARG, "grid_w and grid_h must be equal and non-zero (square grid)");
    if ((uint64_t)cfg->grid_w * cfg->grid_h > 0x7fffffffull) return fail(nullptr, SLAMRS_E_INVALID_ARG, "grid too large");
    if (!(cfg->resolution > 0.0f)) return fail(nullptr, SLAMRS_E_INVALID_ARG, "resolution must be positive");
    if (cfg->rng_mode > SLAMRS_RNG_CALLER) return fail(nullptr, SLAMRS_E_INVALID_ARG, "unknown rng_mode");
    if (!(cfg->resample_threshold >= 0.0f && cfg->resample_threshold <= 1.0f))
        return fail(nullptr, SLAMRS_E_INVALID_ARG, "resample_threshold must be 0 (always resample) or in (0, 1]");
    if (model->kind > SLAMRS_SENSOR_LIKELIHOOD_FIELD) return fail(nullptr, SLAMRS_E_INVALID_ARG, "unknown sensor model kind");
    const bool field = model->kind == SLAMRS_SENSOR_LIKELIHOOD_FIELD;
    if (field) {
        if (!(model->sigma > 0.0f) || !isfinite(model->sigma))
            return fail(nullptr, SLAMRS_E_INVALID_ARG, "sigma must be a positive finite number of metres");
        if (!(model->z_rand > 0.0f && model->z_rand < 1.0f))
            return fail(nullptr, SLAMRS_E_INVALID_ARG, "z_rand must lie in (0, 1)");
        if (!(model->occupied_above >= 0.5f && model->occupied_above < 1.0f))
            return fail(nullptr, SLAMRS_E_INVALID_ARG, "occupied_above must lie in [0.5, 1)");
    }
    const size_t n_cells = (size_t)cfg->grid_w * cfg->grid_h;
    for (size_t i = 0; i < n_cells; ++i)
        if (!(map_probability[i] >= 0.0 && map_probability[i] <= 1.0))
            return fail(nullptr, SLAMRS_E_INVALID_ARG,
                        "map_probability[" + std::to_string(i) + "] is NaN or outside [0, 1]");

    int n_dev = 0;
    if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev == 0) {
        cudaGetLastError();
        return fail(nullptr, SLAMRS_E_NO_DEVICE, "no CUDA device visible; this library has no CPU fallback");
    }
    int device = cfg->device;
    if (device < 0) cudaGetDevice(&device);
    if (device >= n_dev) return fail(nullptr, SLAMRS_E_INVALID_ARG, "device ordinal out of range");

    slamrs_gpu_handle* h = new (std::nothrow) slamrs_gpu_handle();
    if (!h) return fail(nullptr, SLAMRS_E_OUT_OF_MEMORY, "host allocation failed");
    h->cfg = *cfg;
    h->localizer = true;
    h->device = device;
    h->n_total = h->n_local = (uint32_t)cfg->n_particles;
    h->n_cells = (uint32_t)n_cells;
    h->geom = make_map_geom(cfg->pos_x, cfg->pos_y, cfg->resolution, cfg->grid_w, cfg->grid_h);
    h->loc_outside = field ? log((double)model->z_rand) : 0.0;   // ln(z_rand) / the reference's ln(1) for off-grid endpoints

#define CREATE_CU(expr)                                                                                   \
    do {                                                                                                  \
        cudaError_t _e = (expr);                                                                          \
        if (_e != cudaSuccess) {                                                                          \
            const int _code = (_e == cudaErrorMemoryAllocation) ? SLAMRS_E_OUT_OF_MEMORY : SLAMRS_E_CUDA; \
            g_create_error = std::string(#expr) + ": " + cudaGetErrorString(_e);                          \
            cudaGetLastError();                                                                           \
            cudaFree(scratch);                                                                            \
            free_all(h);                                                                                  \
            return _code;                                                                                 \
        }                                                                                                 \
    } while (0)

    uint32_t* scratch = nullptr;   // the distance transform's column pass (freed before returning)
    DeviceGuard guard(device);
    cudaDeviceProp prop;
    CREATE_CU(cudaGetDeviceProperties(&prop, device));
    h->num_sms = prop.multiProcessorCount;
    if (prop.major < 10) {
        g_create_error = "this library is built for sm_100a (B200) only";
        free_all(h);
        return SLAMRS_E_NO_DEVICE;
    }
    CREATE_CU(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
    CREATE_CU(configure_kernels());
    // [ParticleResult x n | StepCounters], zeroed
    h->off_counters = (sizeof(ParticleResult) * (size_t)h->n_total + 255) & ~(size_t)255;
    const size_t pool_bytes = h->off_counters + sizeof(StepCounters);
    CREATE_CU(cudaMalloc(&h->d_pool, pool_bytes));
    CREATE_CU(cudaMemsetAsync(h->d_pool, 0, pool_bytes, h->stream));
    h->d_results_base = h->d_results = (ParticleResult*)h->d_pool;
    h->d_counters = (StepCounters*)((char*)h->d_pool + h->off_counters);
    for (int i = 0; i < 2; ++i) {
        CREATE_CU(cudaMalloc(&h->d_pose[i], sizeof(float) * 3 * h->n_total));
        CREATE_CU(cudaMemsetAsync(h->d_pose[i], 0, sizeof(float) * 3 * h->n_total, h->stream));  // Pose::default()
    }
    CREATE_CU(cudaMalloc(&h->d_wnorm, sizeof(double) * h->n_total));
    CREATE_CU(cudaMalloc(&h->d_cum, sizeof(double) * h->n_total));
    CREATE_CU(cudaMalloc(&h->d_idx, sizeof(uint32_t) * h->n_total));
    CREATE_CU(cudaMalloc(&h->d_fold, sizeof(double) * weights_scratch_doubles()));
    if (cfg->resample_threshold > 0.0f) CREATE_CU(cudaMalloc(&h->d_carry, sizeof(double) * h->n_total));
    CREATE_CU(cudaMemsetAsync(h->d_wnorm, 0, sizeof(double) * h->n_total, h->stream));
    CREATE_CU(cudaMemsetAsync(h->d_idx, 0, sizeof(uint32_t) * h->n_total, h->stream));
    if (cfg->rng_mode == SLAMRS_RNG_CALLER) {
        CREATE_CU(cudaMalloc(&h->d_z, sizeof(double) * 2 * h->n_total));
        CREATE_CU(cudaMalloc(&h->d_u, sizeof(double)));
    }
    CREATE_CU(cudaMallocHost(&h->h_counters, sizeof(StepCounters)));
    memset(h->h_counters, 0, sizeof(StepCounters));
    // d_export: the map's upload buffer here, sim_scan's segment scratch later (as on a SLAM handle)
    CREATE_CU(cudaMalloc(&h->d_export, sizeof(double) * n_cells));
    CREATE_CU(cudaMemcpyAsync(h->d_export, map_probability, sizeof(double) * n_cells, cudaMemcpyHostToDevice, h->stream));
    CREATE_CU(cudaMalloc(&h->d_loc_terms, sizeof(double) * n_cells));
    if (field) CREATE_CU(cudaMalloc(&scratch, sizeof(uint32_t) * n_cells));
    CREATE_CU(launch_loc_terms(h->stream, h->d_export, cfg->grid_w, field ? 1 : 0, model->sigma, model->z_rand,
                               model->occupied_above, cfg->resolution, scratch, h->d_loc_terms));
    h->launches += field ? 2 : 1;
    CREATE_CU(cudaStreamSynchronize(h->stream));
    cudaFree(scratch);
#undef CREATE_CU
    *out = h;
    return SLAMRS_OK;
}

int slamrs_gpu_get_sensor_terms(slamrs_gpu_handle* h, double* out_cells) {
    if (!h || !out_cells) return SLAMRS_E_INVALID_ARG;
    if (!h->localizer) return fail(h, SLAMRS_E_INVALID_ARG, "a SLAM handle has no sensor-term table (only a localizer has one)");
    DeviceGuard g(h->device);
    CU_TRY(h, cudaMemcpyAsync(out_cells, h->d_loc_terms, sizeof(double) * h->n_cells, cudaMemcpyDeviceToHost, h->stream));
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    return SLAMRS_OK;
}

int slamrs_gpu_set_scan_match(slamrs_gpu_handle* h, const slamrs_gpu_scan_match* m) {
    if (!h) return SLAMRS_E_INVALID_ARG;
    if (h->localizer) return fail(h, SLAMRS_E_INVALID_ARG, "a localizer does not scan-match");
    if (!m) {
        h->match_on = false;
        return SLAMRS_OK;
    }
    if (m->struct_size != sizeof(slamrs_gpu_scan_match))
        return fail(h, SLAMRS_E_INVALID_ARG, "slamrs_gpu_scan_match struct_size mismatch");
    if (m->radius > 2u) return fail(h, SLAMRS_E_INVALID_ARG, "scan match radius must be 0, 1 or 2 cells");
    if (!(m->step_xy > 0.0f) || !isfinite(m->step_xy))
        return fail(h, SLAMRS_E_INVALID_ARG, "scan match step_xy must be a positive finite number of metres");
    if (!(m->step_theta > 0.0f) || !isfinite(m->step_theta))
        return fail(h, SLAMRS_E_INVALID_ARG, "scan match step_theta must be a positive finite number of radians");
    if (m->levels < 1u || m->levels > 8u) return fail(h, SLAMRS_E_INVALID_ARG, "scan match levels must lie in 1..8");
    if (m->max_moves < 1u || m->max_moves > 1024u)
        return fail(h, SLAMRS_E_INVALID_ARG, "scan match max_moves must lie in 1..1024");
    if (!h->d_match_stats) {
        DeviceGuard g(h->device);
        CU_TRY(h, cudaMalloc(&h->d_match_stats, sizeof(uint2) * h->n_local));
    }
    h->match = ScanMatchParams{m->radius, m->step_xy, m->step_theta, m->levels, m->max_moves};
    h->match_on = true;
    return SLAMRS_OK;
}

int slamrs_gpu_get_scan_match_stats(slamrs_gpu_handle* h, uint64_t out[4]) {
    if (!h || !out) return SLAMRS_E_INVALID_ARG;
    out[0] = out[1] = out[2] = out[3] = 0;
    if (!h->match_last_step) return SLAMRS_OK;
    DeviceGuard g(h->device);
    std::vector<uint2> per(h->n_local);
    CU_TRY(h, cudaMemcpyAsync(per.data(), h->d_match_stats, sizeof(uint2) * h->n_local, cudaMemcpyDeviceToHost, h->stream));
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    for (const uint2& v : per) {
        out[0] += v.x > 0u;
        out[1] += v.x;
        out[2] += v.y;
        out[3] += v.x == h->match_last_max_moves;
    }
    return SLAMRS_OK;
}

void slamrs_gpu_destroy(slamrs_gpu_handle* h) {
    if (h && getenv("SLAMRS_RAY_TRACE_PRINT")) {
        unsigned long long tr[18];
        DeviceGuard g(h->device);
        cudaStreamSynchronize(h->stream);
        if (ray_trace(tr) == 0) {
            fprintf(stderr, "ray trace: items fused %llu in-place %llu; cycles pop %llu setup %llu walk %llu fused_total %llu wait %llu inplace_wb %llu\n",
                    tr[16], tr[17], tr[0], tr[1], tr[2], tr[3], tr[4], tr[5]);
            fprintf(stderr, "ray trace raw:");
            for (int k = 0; k < 18; ++k) fprintf(stderr, " [%d]%llu", k, tr[k]);
            fprintf(stderr, "\n");
        }
    }
    free_all(h);
}

int slamrs_gpu_upload_scan(slamrs_gpu_handle* h, const float* angle, const float* dist, const uint8_t* valid,
                           uint32_t n_beams) {
    if (!h) return SLAMRS_E_INVALID_ARG;
    if (n_beams > 0 && (!angle || !dist || !valid)) return fail(h, SLAMRS_E_INVALID_ARG, "null scan array");
    if (n_beams > 65535u) return fail(h, SLAMRS_E_INVALID_ARG, "at most 65535 beams per scan");
    DeviceGuard g(h->device);
    int rc = ensure_beam_capacity(h, n_beams ? n_beams : 1);
    if (rc) return rc;
    if (n_beams) {
        // one asynchronous copy out of page-locked memory instead of three staged ones out of the caller's arrays
        if (h->scan_upload_pending) CU_TRY(h, cudaEventSynchronize(h->ev_scan_uploaded));   // the staging buffer is free again
        const size_t cap = h->beam_cap;
        memcpy(h->h_scan_stage, angle, sizeof(float) * n_beams);
        memcpy(h->h_scan_stage + 4u * cap, dist, sizeof(float) * n_beams);
        memcpy(h->h_scan_stage + 8u * cap, valid, n_beams);
        CU_TRY(h, cudaMemcpyAsync(h->d_angle, h->h_scan_stage, 8u * cap + n_beams, cudaMemcpyHostToDevice, h->stream));
        CU_TRY(h, cudaEventRecord(h->ev_scan_uploaded, h->stream));
        h->scan_upload_pending = true;
    }
    h->n_beams = n_beams;
    h->scan_external = false;
    h->order_valid = false;
    // window radius for the ray kernel: farthest measurement, in cells, plus the two extra steps of
    // apply_measurement (map.rs:97) and the slack that lets the ray kernel prove, per ray, that no cell
    // leaves the window (see ray_walk_packed). A non-finite distance still casts a ray, to the grid
    // border: its reach is unbounded, which selects the unfused ray update (cells outside the window take
    // the global-atomic path there; the fused update can only park a bounded number of them).
    float maxd = 0.0f;
    for (uint32_t i = 0; i < n_beams; ++i) {
        const float d = fabsf(dist[i]);
        if (!isfinite(d)) { maxd = INFINITY; break; }
        if (d > maxd) maxd = d;
    }
    const float cells = ceilf(maxd / h->geom.res);
    h->radius_cells = (cells < 4096.0f ? (int)cells : 4096) + 6;
    return SLAMRS_OK;
}

int slamrs_gpu_set_scan_device(slamrs_gpu_handle* h, const float* angle_device, const float* dist_device,
                               const uint8_t* valid_device, uint32_t n_beams, float max_dist) {
    if (!h) return SLAMRS_E_INVALID_ARG;
    if (n_beams > 0 && (!angle_device || !dist_device || !valid_device)) return fail(h, SLAMRS_E_INVALID_ARG, "null scan array");
    if (n_beams > 65535u) return fail(h, SLAMRS_E_INVALID_ARG, "at most 65535 beams per scan");
    h->ext_angle = angle_device; h->ext_dist = dist_device; h->ext_valid = valid_device;
    h->n_beams = n_beams;
    h->scan_external = true;
    h->order_valid = false;
    // max_dist bounds |distance| over the scan; +inf, NaN or <= 0 mean "unknown": the unfused ray update, which
    // takes any scan (see slamrs_gpu.h)
    const float cells = max_dist > 0.0f ? ceilf(max_dist / h->geom.res) : INFINITY;
    h->radius_cells = ((cells == cells && cells < 4096.0f) ? (int)cells : 4096) + 6;
    return SLAMRS_OK;
}

int slamrs_gpu_step_async(slamrs_gpu_handle* h, float dist_left, float dist_right, float wheel_dist,
                          const double* z_draws, const double* resample_u) {
    if (!h) return SLAMRS_E_INVALID_ARG;
    const bool caller = h->cfg.rng_mode == SLAMRS_RNG_CALLER;
    if (caller && (!z_draws || !resample_u))
        return fail(h, SLAMRS_E_INVALID_ARG, "rng_mode CALLER needs z_draws and resample_u");
    DeviceGuard g(h->device);
    cudaStream_t s = h->stream;
    const OdomModel od = odometry_new(dist_left, dist_right, wheel_dist);
    if (caller) {
        CU_TRY(h, cudaMemcpyAsync(h->d_z, z_draws, sizeof(double) * 2 * h->n_total, cudaMemcpyHostToDevice, s));
        CU_TRY(h, cudaMemcpyAsync(h->d_u, resample_u, sizeof(double), cudaMemcpyHostToDevice, s));
    }
    if (h->localizer) return loc_step_async(h, od, caller);
    // beam order for the ray kernel (side stream, concurrent with the likelihood kernel); scans with
    // more beams than the sort handles keep scan order
    const bool sorted = h->n_beams > 32u && h->n_beams <= SORT_MAX_BEAMS;
    const ScanDevice scan = h->scan_external
                                ? ScanDevice{h->ext_angle, h->ext_dist, h->ext_valid, h->n_beams, sorted ? h->d_order : nullptr}
                                : ScanDevice{h->d_angle, h->d_dist, h->d_valid, h->n_beams, sorted ? h->d_order : nullptr};
    if (sorted && !h->order_valid) {
        // everything issued so far (scan upload, the previous step's ray kernel that still reads the old
        // order) precedes the sort
        CU_TRY(h, cudaEventRecord(h->ev_indices, s));
        CU_TRY(h, cudaStreamWaitEvent(h->side_stream, h->ev_indices, 0));
        launch_sort_beams(h->side_stream, scan.dist, h->n_beams, h->d_order);
        CU_TRY(h, cudaEventRecord(h->ev_sort, h->side_stream));
        h->launches++;
        h->order_valid = true;
        h->order_pending = true;
    }
    if (h->profiling && h->prof_recorded == PROF_RING) {
        int prc = prof_flush(h);
        if (prc) return prc;
    }
    const int cur = h->cur, nxt = cur ^ 1;
    const size_t grid_bytes = h->cells_per_grid * sizeof(uint32_t);
    const bool all_particles = (h->cfg.flags & SLAMRS_FLAG_UPDATE_ALL_PARTICLES) != 0;
    const uint32_t res_off = (uint32_t)(h->step & 1ull) * h->n_total;
    h->d_results = h->d_results_base + res_off;

    const bool force_generic = (h->cfg.flags & SLAMRS_FLAG_GENERIC_RAY_KERNEL) != 0;
    const bool fuse = h->defer && !all_particles &&
                      ray_update_can_fuse(h->geom, h->n_beams, h->cells_per_grid, force_generic, h->radius_cells);
    // per-slot reader / done counters and per-item hand-over flags of the ray update (off the critical path: long before their use)
    const bool half_items = ray_update_can_fuse(h->geom, h->n_beams, h->cells_per_grid, force_generic, h->radius_cells);
    // Pulls without a second barrier (world > 1, default path): the ray update publishes, per integrated slot, that the
    // slot is complete; the pull kernels run on the side stream behind the planner, wait per source for that mark and
    // overlap the tail of the ray update. Every rank takes the same decision (same configuration, same scan).
    const bool flag_pulls = h->world > 1 && fuse && half_items && h->boxed_copy && h->p2p_exchange;
    const uint32_t pull_epoch = flag_pulls ? (uint32_t)(h->step + 1ull) : 0u;
    // (readers | done | xflag | xdone are cleared by k_motion)
    const size_t n_zero = half_items ? 2 * (size_t)h->n_slots + 2 * (size_t)h->n_local : 0;
    // 1. motion sample + beam-endpoint likelihood (pre-update map) -> results[first .. first+n_local)
    PROF_MARK(h, 0);
    launch_motion_likelihood(s, h->geom, od, scan, h->d_pose[cur], h->d_slot[cur], h->defer ? h->d_alias : nullptr, h->d_cells, h->d_meta, h->cells_per_grid,
                             h->d_results, h->first, h->n_local, caller ? h->d_z : nullptr, h->cfg.seed, h->step, h->d_term_table, h->d_valid_list, h->d_n_valid,
                             h->d_carry, h->d_counters, h->p2p_exchange ? h->d_peer_results : nullptr, res_off, h->rank, h->world,
                             h->d_readers, (uint32_t)n_zero, h->match_on ? &h->match : nullptr, h->d_match_stats);
    h->launches += h->match_on ? 3 : 2;   // k_motion (+ k_scan_match) + k_likelihood
    h->match_last_step = h->match_on;
    h->match_last_max_moves = h->match.max_moves;
    // 2. the one exchange step: every GPU needs every particle's weight, pose and slot. Default:
    //    k_likelihood has already stored each record into every peer (NVLink), only the barrier is
    //    left. SLAMRS_FLAG_NCCL_EXCHANGE: ncclAllGather of the shard instead.
    PROF_MARK(h, 1);
    if (h->world > 1) {
        if (h->p2p_exchange) {
            int brc = step_barrier(h);
            if (brc) return brc;
        } else {
            std::string err;
            if (comm_all_gather(h->comm, h->d_results + h->first, h->d_results, sizeof(ParticleResult) * h->n_local, s, &err))
                return fail(h, SLAMRS_E_NCCL, err);
        }
    }
    // 3. normalise, argmax, running sum; systematic resampling indices (replicated on every GPU);
    //    which local particles survive
    PROF_MARK(h, 2);
    // (k_weights also zeroes the per-step counters)
    launch_weights(s, h->d_results, h->n_total, h->d_wnorm, h->d_cum, h->d_fold, (double)h->cfg.resample_threshold, h->d_counters);
    // 3b. deferred copies: the clones among the particles about to be written get their own cells. Either the
    //     ray kernel does it while it integrates the scan (fused: k_resample_indices lists the survivors as
    //     clones | owners, no copy kernels), or they are listed now and copied after PROF_MARK 3. Before the
    //     planner starts: both write the alias table.
    RayLists ray{nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, 0u, 0u};
    if (fuse) ray = RayLists{h->d_ray_items, h->d_ray_items + h->n_local, h->d_slot[cur], h->d_alias, h->d_readers, h->d_meta,
                             h->n_local, flag_pulls ? 1u : 0u};
    launch_resample_indices(s, h->d_results, h->d_cum, h->n_total, caller ? h->d_u : nullptr, h->cfg.seed, h->step,
                            h->d_idx, h->d_pose[nxt], h->first, h->n_local, !all_particles, h->d_alive, ray, h->d_wnorm, h->d_carry,
                            h->d_counters);
    if (all_particles) {
        launch_mark_alive(s, h->d_idx, h->n_total, h->first, h->n_local, true, h->d_alive, h->d_counters);
        h->launches++;
    }
    if (h->defer && !fuse) {
        if (all_particles)   // every clone: ordered list with fan-out sub-runs
            launch_materialize_list(s, nullptr, h->n_total, h->first, h->n_local, h->d_slot[cur], h->d_alias, h->d_cells,
                                    h->cells_per_grid, h->d_meta, h->d_bands, h->n_bands, h->d_mat_items, h->d_mat_leaders,
                                    h->d_mat_roots, h->d_counters);
        else                 // the clones among the survivors: a few hundred, listed in parallel
            launch_materialize_alive(s, h->d_alive, h->n_local, h->d_slot[cur], h->d_alias, h->d_cells, h->cells_per_grid,
                                     h->d_meta, h->d_bands, h->n_bands, h->d_mat_items, h->d_counters);
        h->launches++;
    }
    // 4. plan (side stream): which grids stay, which are duplicated locally, which are pulled from a
    //    peer. It needs only the index vector, so it runs concurrently with the ray update.
    CU_TRY(h, cudaEventRecord(h->ev_indices, s));
    CU_TRY(h, cudaStreamWaitEvent(h->side_stream, h->ev_indices, 0));
    PlanArgs pa{};
    pa.results = h->d_results;
    pa.idx = h->d_idx;
    pa.n_total = h->n_total; pa.n_local = h->n_local; pa.rank = h->rank; pa.world = h->world;
    pa.slot_old = h->d_slot[cur]; pa.slot_new = h->d_slot[nxt];
    pa.keep = h->d_keep; pa.need = h->d_need; pa.free_list = h->d_free; pa.spare_list = h->d_spare;
    pa.n_spare_cap = h->n_spare;
    pa.copies = h->d_copies; pa.leaders = h->d_leaders;
    pa.cells = h->d_cells; pa.cells_per_grid = h->cells_per_grid;
    pa.peer_cells = h->d_peer_cells;
    pa.meta = h->d_meta; pa.peer_meta = h->d_peer_meta;
    pa.bands = h->d_bands; pa.peer_bands = h->d_peer_bands; pa.n_bands = h->n_bands;
    pa.counters = h->d_counters;
    pa.history = h->d_history;
    pa.step = h->step;
    pa.staged = plan_can_stage(h->n_local, h->n_spare);
    pa.alias_of = h->d_alias; pa.defer = h->defer;
    launch_plan(h->side_stream, pa);
    h->launches += 3;   // k_weights, k_resample_indices, k_plan
    if (flag_pulls) {
        // the first uses of remote sources, a short list: each job waits for its source's owner (NVLink reads)
        launch_pull(h->side_stream, h->d_copies, h->d_leaders, &h->d_counters->n_copies, &h->d_counters->n_leaders,
                    h->n_local, h->geom, h->d_counters, h->num_sms, pull_epoch, h->barrier_timeout_ns, h->d_meta, h->d_readers,
                    h->d_readers + h->n_slots);
        h->launches++;
    }
    CU_TRY(h, cudaEventRecord(h->ev_plan, h->side_stream));
    PROF_MARK(h, 3);
    if (h->defer && !fuse) {
        int mrc = materialize_copies(h, all_particles);
        if (mrc) return mrc;
    }
    // 5. integrate the scan into the grids that survive resampling (all grids in strict mode)
    PROF_MARK(h, 4);
    if (h->order_pending) {
        CU_TRY(h, cudaStreamWaitEvent(s, h->ev_sort, 0));
        h->order_pending = false;
    }
    CU_TRY(h, launch_ray_update(s, h->geom, scan, h->d_results, h->first, h->n_local, h->d_alive,
                                fuse ? h->d_ray_items : nullptr, fuse ? h->d_ray_items + h->n_local : nullptr,
                                fuse ? h->d_readers : nullptr,
                                fuse ? h->d_readers + h->n_slots : nullptr, h->d_readers + 2 * (size_t)h->n_slots, h->d_ray_xchg,
                                h->d_ray_spill, h->d_slot[cur],
                                h->d_cells, h->d_meta, h->d_bands, h->cells_per_grid, h->radius_cells, h->d_counters, &h->window_cells,
                                force_generic, h->num_sms, h->d_readers + 2 * (size_t)h->n_slots + h->n_local, pull_epoch));
    h->launches++;
    PROF_MARK(h, 5);
    CU_TRY(h, cudaStreamWaitEvent(s, h->ev_plan, 0));   // join: the copy lists are ready
    // 6. grid traffic: one launch copies from local and (over NVLink) remote sources alike. Across
    //    GPUs one barrier first: every source grid, wherever it lives, has received the scan. No
    //    second barrier: nothing written in this step is a slot a peer reads in this step (k_plan).
    if (h->world > 1 && !flag_pulls) {
        int brc = step_barrier(h);
        if (brc) return brc;
    }
    PROF_MARK(h, 6);
    if ((h->defer && h->world == 1) || flag_pulls) {
        // deferred copies on one GPU: the planner's list is empty (no remote sources), nothing to launch
    } else if (h->boxed_copy) {
        // deferred copies: what is left here are the first uses of remote sources, a short list
        launch_copy_boxed(s, h->d_copies, h->d_leaders, &h->d_counters->n_copies, &h->d_counters->n_leaders, h->n_local,
                          h->d_jobs, h->geom, h->d_counters, h->num_sms, h->defer);
        h->launches++;
    } else {
        launch_copy(s, h->d_copies, h->d_leaders, &h->d_counters->n_copies, &h->d_counters->n_leaders, h->cells_per_grid,
                    h->num_sms);
        launch_account_full_copy(s, &h->d_counters->n_copies, &h->d_counters->n_leaders, grid_bytes, h->d_counters);
        h->launches++;
    }
    if (!((h->defer && h->world == 1) || flag_pulls)) h->launches++;
    PROF_MARK(h, 7);
    // (deferred copies on one GPU: the list is empty, the kernel only completes the step's history record)
    launch_commit_boxes(s, h->d_copies, &h->d_counters->n_copies, (h->defer && h->world == 1) ? 1u : h->n_local, h->geom,
                        h->boxed_copy, h->d_counters, h->d_history + (h->step % STEP_HISTORY),
                        h->mirror_wanted ? h->h_counters : nullptr);   // (a store over PCIe: only when a sync follows at once)
    h->launches++;
    if (h->profiling) h->prof_recorded++;
    CU_TRY(h, cudaGetLastError());
    h->cur = nxt;
    h->step++;
    h->counters_fresh = false;
    h->mirror_by_step = h->mirror_wanted;
    h->est_box_stale = false;
    return SLAMRS_OK;
}

int slamrs_gpu_sync(slamrs_gpu_handle* h) {
    if (!h) return SLAMRS_E_INVALID_ARG;
    DeviceGuard g(h->device);
    int rc = fetch_counters(h);
    if (rc) return rc;
    if (h->h_counters->barrier_timeout)
        return fail(h, SLAMRS_E_INTERNAL,
                    h->h_counters->barrier_timeout == 2ull
                        ? "a peer GPU's handle was destroyed (its step failed or its owner left); this handle can only be destroyed"
                        : "a peer GPU did not reach the step barrier within the time limit");
    if (h->h_counters->fuse_overflow)
        return fail(h, SLAMRS_E_INTERNAL, "fused ray update: more window-bypassing hits than its scratch holds");
    if (h->h_counters->window_overflow)
        return fail(h, SLAMRS_E_WINDOW,
                    "a particle's informed extent outgrew its windowed grid slot; raise slot_cells (the scan was not "
                    "integrated into that grid)");
    if (h->h_counters->staging_short)
        return fail(h, SLAMRS_E_STAGING,
                    "cross-GPU migration needed more free grid slots than available; raise spare_slots");
    return SLAMRS_OK;
}

int slamrs_gpu_update(slamrs_gpu_handle* h, const float* angle, const float* dist, const uint8_t* valid,
                      uint32_t n_beams, float dist_left, float dist_right, float wheel_dist, const double* z_draws,
                      const double* resample_u) {
    int rc = slamrs_gpu_upload_scan(h, angle, dist, valid, n_beams);
    if (rc) return rc;
    h->mirror_wanted = true;   // the step's last kernel leaves the counters in the host mirror: the sync below launches nothing
    rc = slamrs_gpu_step_async(h, dist_left, dist_right, wheel_dist, z_draws, resample_u);
    h->mirror_wanted = false;
    if (rc) return rc;
    return slamrs_gpu_sync(h);
}

int slamrs_gpu_pose(slamrs_gpu_handle* h, float out_xyt[3]) {
    if (!h || !out_xyt) return SLAMRS_E_INVALID_ARG;
    DeviceGuard g(h->device);
    int rc = fetch_counters(h);
    if (rc) return rc;
    out_xyt[0] = h->h_counters->est_pose[0];
    out_xyt[1] = h->h_counters->est_pose[1];
    out_xyt[2] = h->h_counters->est_pose[2];
    return SLAMRS_OK;
}

namespace {
// exports [x0,x1) x [y0,y1) of the estimate's grid in `format` into the caller's host buffer; pipelined: the copy
// runs on the handle's copy stream and the call returns once it is queued (slamrs_gpu_map_wait waits for it)
int export_window(slamrs_gpu_handle* h, uint32_t format, int x0, int y0, int x1, int y1, void* out, bool pipelined = false) {
    if (format > SLAMRS_MAP_U8) return fail(h, SLAMRS_E_INVALID_ARG, "unknown map format");
    if (x0 < 0 || y0 < 0 || x1 > (int)h->geom.gw || y1 > (int)h->geom.gh || x1 < x0 || y1 < y0)
        return fail(h, SLAMRS_E_INVALID_ARG, "map window outside the grid");
    const size_t n = (size_t)(x1 - x0) * (size_t)(y1 - y0);
    if (n == 0 && h->world == 1) return SLAMRS_OK;
    const size_t bytes = n * (format == SLAMRS_MAP_F64 ? 8u : (format == SLAMRS_MAP_F32 ? 4u : 1u));
    cudaStream_t s = h->stream;
    if (h->world > 1) {
        // The estimate's grid lives on one GPU. After a barrier (its step, pulls included, is complete) the rank
        // that asked converts it straight out of the owner's pool over NVLink: no broadcast, one D2H copy.
        int rc = fetch_counters(h);  // owner of the estimate, identical on every rank
        if (rc) return rc;
        rc = step_barrier(h);
        if (rc) return rc;
        if (out == nullptr) return SLAMRS_OK;   // took part, does not want the map
    }
    double* dst = h->d_export;
    int k = 0;
    if (pipelined) {
        k = h->async_next;
        h->async_next ^= 1;
        if (h->async_pending[k]) CU_TRY(h, cudaStreamWaitEvent(s, h->ev_copied[k], 0));   // the buffer's previous copy has left it
        dst = h->d_export_async[k];
    }
    if (h->world > 1) {
        const uint32_t owner = (uint32_t)h->h_counters->est_owner;
        launch_export(s, h->host_peer_cells[owner], h->host_peer_meta[owner], h->cells_per_grid, h->peer_counters[owner], h->geom,
                      x0, y0, x1, y1, (int)format, dst);
    } else {
        launch_export(s, h->d_cells, h->d_meta, h->cells_per_grid, h->d_counters, h->geom, x0, y0, x1, y1, (int)format, dst);
    }
    h->launches++;
    if (pipelined) {
        CU_TRY(h, cudaEventRecord(h->ev_exported[k], s));
        CU_TRY(h, cudaStreamWaitEvent(h->copy_stream, h->ev_exported[k], 0));
        CU_TRY(h, cudaMemcpyAsync(out, dst, bytes, cudaMemcpyDeviceToHost, h->copy_stream));
        CU_TRY(h, cudaEventRecord(h->ev_copied[k], h->copy_stream));
        h->async_pending[k] = true;
        return SLAMRS_OK;
    }
    CU_TRY(h, cudaMemcpyAsync(out, h->d_export, bytes, cudaMemcpyDeviceToHost, s));
    CU_TRY(h, cudaStreamSynchronize(s));
    CU_TRY(h, cudaGetLastError());
    return SLAMRS_OK;
}
}  // namespace

int slamrs_gpu_map_probability(slamrs_gpu_handle* h, double* out_cells) {
    if (!h || (!out_cells && h->world == 1)) return SLAMRS_E_INVALID_ARG;
    if (h->localizer) return fail(h, SLAMRS_E_INVALID_ARG, NO_GRIDS);
    DeviceGuard g(h->device);
    return export_window(h, SLAMRS_MAP_F64, 0, 0, (int)h->geom.gw, (int)h->geom.gh, out_cells);
}

int slamrs_gpu_map_probability_async(slamrs_gpu_handle* h, double* out_cells) {
    if (!h || (!out_cells && h->world == 1)) return SLAMRS_E_INVALID_ARG;
    if (h->localizer) return fail(h, SLAMRS_E_INVALID_ARG, NO_GRIDS);
    DeviceGuard g(h->device);
    return export_window(h, SLAMRS_MAP_F64, 0, 0, (int)h->geom.gw, (int)h->geom.gh, out_cells, true);
}

int slamrs_gpu_map_wait(slamrs_gpu_handle* h) {
    if (!h) return SLAMRS_E_INVALID_ARG;
    DeviceGuard g(h->device);
    for (int k = 0; k < 2; ++k) {
        if (!h->async_pending[k]) continue;
        CU_TRY(h, cudaEventSynchronize(h->ev_copied[k]));
        h->async_pending[k] = false;
    }
    CU_TRY(h, cudaGetLastError());
    return SLAMRS_OK;
}

int slamrs_gpu_map_extent(slamrs_gpu_handle* h, int32_t out_x0y0x1y1[4]) {
    if (!h || !out_x0y0x1y1) return SLAMRS_E_INVALID_ARG;
    if (h->localizer) return fail(h, SLAMRS_E_INVALID_ARG, NO_GRIDS);
    DeviceGuard g(h->device);
    if (h->world == 1 && h->step > 0 && !h->est_box_stale) {   // the step left the extent of the published map in the counters
        int rc = fetch_counters(h);
        if (rc) return rc;
        for (int i = 0; i < 4; ++i) out_x0y0x1y1[i] = h->h_counters->est_box[i];
        return SLAMRS_OK;
    }
    cudaStream_t s = h->stream;
    int* d4 = reinterpret_cast<int*>(h->d_export);
    if (h->world > 1) {
        int rc = fetch_counters(h);
        if (rc) return rc;
        rc = step_barrier(h);
        if (rc) return rc;
        const uint32_t owner = (uint32_t)h->h_counters->est_owner;
        launch_estimate_extent(s, h->host_peer_meta[owner], h->peer_counters[owner], d4);
    } else {
        launch_estimate_extent(s, h->d_meta, h->d_counters, d4);
    }
    h->launches++;
    CU_TRY(h, cudaMemcpyAsync(out_x0y0x1y1, d4, 4 * sizeof(int), cudaMemcpyDeviceToHost, s));
    CU_TRY(h, cudaStreamSynchronize(s));
    return SLAMRS_OK;
}

int slamrs_gpu_map_window(slamrs_gpu_handle* h, uint32_t format, int32_t x0, int32_t y0, int32_t x1, int32_t y1,
                          void* out) {
    if (!h || (!out && h->world == 1)) return SLAMRS_E_INVALID_ARG;
    if (h->localizer) return fail(h, SLAMRS_E_INVALID_ARG, NO_GRIDS);
    DeviceGuard g(h->device);
    return export_window(h, format, x0, y0, x1, y1, out);
}

int slamrs_gpu_effective_particles(slamrs_gpu_handle* h, double* out) {
    if (!h || !out) return SLAMRS_E_INVALID_ARG;
    DeviceGuard g(h->device);
    int rc = fetch_counters(h);
    if (rc) return rc;
    *out = h->step == 0 ? (double)h->n_total : h->h_counters->n_eff;   // uniform weights before the first update
    return SLAMRS_OK;
}

int slamrs_gpu_sim_scan(slamrs_gpu_handle* h, const float* segments_xyxy, uint32_t n_segments, const float pose_xyt[3],
                        uint32_t n_beams, float scanner_range, uint32_t* out_n) {
    if (!h || !pose_xyt || (n_segments && !segments_xyxy)) return SLAMRS_E_INVALID_ARG;
    if (n_beams > 65535u) return fail(h, SLAMRS_E_INVALID_ARG, "at most 65535 beams per scan");
    DeviceGuard g(h->device);
    int rc = ensure_beam_capacity(h, n_beams ? n_beams : 1);
    if (rc) return rc;
    cudaStream_t s = h->stream;
    float* d_seg = reinterpret_cast<float*>(h->d_export);              // scratch: 16 bytes per segment
    if ((size_t)n_segments * 16u + 16u > sizeof(double) * (size_t)h->n_cells)
        return fail(h, SLAMRS_E_INVALID_ARG, "too many scene segments for the scratch buffer");
    uint32_t* d_cnt = reinterpret_cast<uint32_t*>(d_seg + 4 * (size_t)n_segments);
    if (n_segments)
        CU_TRY(h, cudaMemcpyAsync(d_seg, segments_xyxy, 16 * (size_t)n_segments, cudaMemcpyHostToDevice, s));
    CU_TRY(h, cudaMemsetAsync(d_cnt, 0, 2 * sizeof(uint32_t), s));
    launch_sim_scan(s, d_seg, n_segments, pose_xyt[0], pose_xyt[1], pose_xyt[2], n_beams, scanner_range, h->d_angle,
                    h->d_dist, h->d_valid, d_cnt);
    h->launches++;
    uint32_t res[2] = {0, 0};
    CU_TRY(h, cudaMemcpyAsync(res, d_cnt, sizeof(res), cudaMemcpyDeviceToHost, s));
    CU_TRY(h, cudaStreamSynchronize(s));
    CU_TRY(h, cudaGetLastError());
    h->n_beams = res[0];
    h->scan_external = false;
    h->order_valid = false;
    float maxd;
    memcpy(&maxd, &res[1], 4);
    const float cells = ceilf(maxd / h->geom.res);
    h->radius_cells = ((cells == cells && cells < 4096.0f) ? (int)cells : 4096) + 6;
    if (out_n) *out_n = res[0];
    return SLAMRS_OK;
}

int slamrs_gpu_get_scan(slamrs_gpu_handle* h, float* out_angle, float* out_dist, uint8_t* out_valid, uint32_t cap,
                        uint32_t* out_n) {
    if (!h || !out_n) return SLAMRS_E_INVALID_ARG;
    if (h->scan_external) return fail(h, SLAMRS_E_INVALID_ARG, "the current scan lives in caller-owned device memory");
    DeviceGuard g(h->device);
    *out_n = h->n_beams;
    const uint32_t n = h->n_beams < cap ? h->n_beams : cap;
    if (n && out_angle) CU_TRY(h, cudaMemcpyAsync(out_angle, h->d_angle, sizeof(float) * n, cudaMemcpyDeviceToHost, h->stream));
    if (n && out_dist) CU_TRY(h, cudaMemcpyAsync(out_dist, h->d_dist, sizeof(float) * n, cudaMemcpyDeviceToHost, h->stream));
    if (n && out_valid) CU_TRY(h, cudaMemcpyAsync(out_valid, h->d_valid, n, cudaMemcpyDeviceToHost, h->stream));
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    return SLAMRS_OK;
}

const char* slamrs_gpu_last_error(const slamrs_gpu_handle* h) { return h ? h->last_error.c_str() : g_create_error.c_str(); }

int slamrs_gpu_get_stats(slamrs_gpu_handle* h, slamrs_gpu_stats* out) {
    if (!h || !out) return SLAMRS_E_INVALID_ARG;
    DeviceGuard g(h->device);
    int rc = fetch_counters(h);
    if (rc) return rc;
    const StepCounters& c = *h->h_counters;
    out->step = h->step;
    out->grids_copied = c.n_copies + c.n_mat;
    out->grids_pulled = c.n_pulls;
    out->distinct_sources = c.distinct;
    out->resample_clamped = c.clamped;
    out->counter_saturated = c.saturated;
    out->spilled_cells = c.spilled;
    out->window_cells = h->window_cells;
    out->particles_integrated = c.n_alive;
    out->bytes_per_grid = h->localizer ? 0 : h->cells_per_grid * sizeof(uint32_t);
    out->window_overflow = c.window_overflow;
    out->copy_bytes = c.copy_bytes;
    out->resample_exact_fallback = c.fold_fallback;
    out->resample_fold_rounds = c.fold_rounds;
    out->resampled = h->step == 0 ? 0 : c.do_resample;
    return SLAMRS_OK;
}

int slamrs_gpu_set_profiling(slamrs_gpu_handle* h, int enabled) {
    if (!h) return SLAMRS_E_INVALID_ARG;
    DeviceGuard g(h->device);
    if (enabled && h->prof_events.empty()) {
        h->prof_events.resize((size_t)PROF_RING * PROF_MARKS);
        for (auto& e : h->prof_events) CU_TRY(h, cudaEventCreate(&e));
    }
    if (!enabled) {
        int rc = prof_flush(h);
        if (rc) return rc;
    }
    h->profiling = enabled != 0;
    return SLAMRS_OK;
}

int slamrs_gpu_get_phase_ms(slamrs_gpu_handle* h, double out_ms[SLAMRS_PHASE_COUNT], uint64_t* out_steps) {
    if (!h || !out_ms || !out_steps) return SLAMRS_E_INVALID_ARG;
    DeviceGuard g(h->device);
    int rc = prof_flush(h);
    if (rc) return rc;
    for (int p = 0; p < SLAMRS_PHASE_COUNT; ++p) { out_ms[p] = h->prof_ms[p]; h->prof_ms[p] = 0.0; }
    *out_steps = h->prof_steps;
    h->prof_steps = 0;
    return SLAMRS_OK;
}

int slamrs_gpu_get_step_history(slamrs_gpu_handle* h, uint64_t first_step, uint32_t count, uint64_t* out_triples) {
    // seven values per step: grids_copied, grids_pulled, distinct_sources, source_reads, particles_integrated,
    // copy_bytes, ray_cell_steps, ray_copy_bytes
    if (!h || !out_triples || count > STEP_HISTORY) return SLAMRS_E_INVALID_ARG;
    if (h->localizer) return fail(h, SLAMRS_E_INVALID_ARG, NO_GRIDS);
    DeviceGuard g(h->device);
    std::vector<StepRecord> ring(STEP_HISTORY);
    CU_TRY(h, cudaMemcpyAsync(ring.data(), h->d_history, sizeof(StepRecord) * STEP_HISTORY, cudaMemcpyDeviceToHost, h->stream));
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    for (uint32_t i = 0; i < count; ++i) {
        const StepRecord& r = ring[(first_step + i) % STEP_HISTORY];
        if (r.step != first_step + i) return fail(h, SLAMRS_E_INVALID_ARG, "step no longer in the history ring");
        uint64_t* o = out_triples + (size_t)SLAMRS_HISTORY_VALUES * i;
        o[0] = r.n_copies; o[1] = r.n_pulls; o[2] = r.distinct; o[3] = r.n_leaders; o[4] = r.n_alive; o[5] = r.copy_bytes;
        o[6] = r.ray_cell_steps; o[7] = r.ray_copy_bytes;
    }
    return SLAMRS_OK;
}

void* slamrs_gpu_stream(slamrs_gpu_handle* h) { return h ? (void*)h->stream : nullptr; }
uint64_t slamrs_gpu_launch_count(const slamrs_gpu_handle* h) { return h ? h->launches : 0; }

int slamrs_gpu_get_poses(slamrs_gpu_handle* h, float* out_xyt) {
    if (!h || !out_xyt) return SLAMRS_E_INVALID_ARG;
    DeviceGuard g(h->device);
    CU_TRY(h, cudaMemcpyAsync(out_xyt, h->d_pose[h->cur], sizeof(float) * 3 * h->n_local, cudaMemcpyDeviceToHost, h->stream));
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    return SLAMRS_OK;
}

int slamrs_gpu_get_slots(slamrs_gpu_handle* h, int32_t* out_slot_of, int32_t* out_spare, uint32_t* out_n_spare) {
    if (!h) return SLAMRS_E_INVALID_ARG;
    if (h->localizer) return fail(h, SLAMRS_E_INVALID_ARG, NO_GRIDS);
    DeviceGuard g(h->device);
    if (out_slot_of)
        CU_TRY(h, cudaMemcpyAsync(out_slot_of, h->d_slot[h->cur], sizeof(int32_t) * h->n_local, cudaMemcpyDeviceToHost, h->stream));
    if (out_spare && h->n_spare)
        CU_TRY(h, cudaMemcpyAsync(out_spare, h->d_spare, sizeof(int32_t) * h->n_spare, cudaMemcpyDeviceToHost, h->stream));
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    if (out_n_spare) *out_n_spare = h->n_spare;
    return SLAMRS_OK;
}

int slamrs_gpu_init_uniform(slamrs_gpu_handle* h, const float box[4]) {
    if (!h || !box) return SLAMRS_E_INVALID_ARG;
    if (!(box[2] >= box[0] && box[3] >= box[1])) return fail(h, SLAMRS_E_INVALID_ARG, "empty box");
    DeviceGuard g(h->device);
    launch_init_uniform(h->stream, h->cfg.seed, h->first, h->n_local, box[0], box[1], box[2], box[3], h->d_pose[h->cur]);
    h->launches++;
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    CU_TRY(h, cudaGetLastError());
    return SLAMRS_OK;
}

int slamrs_gpu_set_poses(slamrs_gpu_handle* h, const float* xyt) {
    if (!h || !xyt) return SLAMRS_E_INVALID_ARG;
    DeviceGuard g(h->device);
    CU_TRY(h, cudaMemcpyAsync(h->d_pose[h->cur], xyt, sizeof(float) * 3 * h->n_local, cudaMemcpyHostToDevice, h->stream));
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    return SLAMRS_OK;
}

int slamrs_gpu_get_weights(slamrs_gpu_handle* h, double* out_norm, double* out_raw) {
    if (!h) return SLAMRS_E_INVALID_ARG;
    DeviceGuard g(h->device);
    if (out_norm)
        CU_TRY(h, cudaMemcpyAsync(out_norm, h->d_wnorm, sizeof(double) * h->n_total, cudaMemcpyDeviceToHost, h->stream));
    if (out_raw)
        CU_TRY(h, cudaMemcpy2DAsync(out_raw, sizeof(double), h->d_results, sizeof(ParticleResult), sizeof(double),
                                    h->n_total, cudaMemcpyDeviceToHost, h->stream));
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    return SLAMRS_OK;
}

int slamrs_gpu_get_resample_indices(slamrs_gpu_handle* h, uint32_t* out_idx) {
    if (!h || !out_idx) return SLAMRS_E_INVALID_ARG;
    DeviceGuard g(h->device);
    CU_TRY(h, cudaMemcpyAsync(out_idx, h->d_idx, sizeof(uint32_t) * h->n_total, cudaMemcpyDeviceToHost, h->stream));
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    return SLAMRS_OK;
}

int slamrs_gpu_get_max_particle(slamrs_gpu_handle* h, uint64_t* out) {
    if (!h || !out) return SLAMRS_E_INVALID_ARG;
    DeviceGuard g(h->device);
    int rc = fetch_counters(h);
    if (rc) return rc;
    *out = h->h_counters->max_particle;
    return SLAMRS_OK;
}

static int local_slot(slamrs_gpu_handle* h, uint64_t particle, int32_t* slot) {
    if (particle < h->first || particle >= (uint64_t)h->first + h->n_local)
        return fail(h, SLAMRS_E_NOT_LOCAL, "particle is owned by another rank");
    CU_TRY(h, cudaMemcpyAsync(slot, h->d_slot[h->cur] + (particle - h->first), sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    return SLAMRS_OK;
}
// the slot whose cells the particle's grid is read from: its own, or its source's while it is an unwritten clone
static int local_root_slot(slamrs_gpu_handle* h, uint64_t particle, int32_t* slot) {
    int rc = local_slot(h, particle, slot);
    if (rc || !h->defer) return rc;
    CU_TRY(h, cudaMemcpyAsync(slot, h->d_alias + *slot, sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    return SLAMRS_OK;
}

int slamrs_gpu_get_cells(slamrs_gpu_handle* h, uint64_t particle, uint32_t* out_cells) {
    if (!h || !out_cells) return SLAMRS_E_INVALID_ARG;
    if (h->localizer) return fail(h, SLAMRS_E_INVALID_ARG, NO_GRIDS);
    DeviceGuard g(h->device);
    int32_t slot = 0;
    int rc = local_root_slot(h, particle, &slot);
    if (rc) return rc;
    // the slot stores its cells tile by tile (or windowed); the export kernel returns them in logical order
    launch_export_slot(h->stream, h->d_cells + (size_t)slot * h->cells_per_grid, h->d_meta + slot, h->geom, false, h->d_export);
    h->launches++;
    CU_TRY(h, cudaMemcpyAsync(out_cells, h->d_export, sizeof(uint32_t) * h->n_cells, cudaMemcpyDeviceToHost, h->stream));
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    return SLAMRS_OK;
}

int slamrs_gpu_set_cells(slamrs_gpu_handle* h, uint64_t particle, const uint32_t* cells) {
    if (!h || !cells) return SLAMRS_E_INVALID_ARG;
    if (h->localizer) return fail(h, SLAMRS_E_INVALID_ARG, NO_GRIDS);
    DeviceGuard g(h->device);
    int32_t slot = 0;
    int rc = unshare_all(h);
    if (rc) return rc;
    rc = local_slot(h, particle, &slot);
    if (rc) return rc;
    // extent of the informed cells of the new image
    const int gw = (int)h->geom.gw, gh = (int)h->geom.gh;
    int x0 = gw, y0 = gh, x1 = -1, y1 = -1;
    for (int y = 0; y < gh; ++y) {
        const uint32_t* row = cells + (size_t)y * gw;
        int fx = -1, lx = -1;
        for (int x = 0; x < gw; ++x)
            if (row[x]) { if (fx < 0) fx = x; lx = x; }
        if (fx >= 0) {
            if (fx < x0) x0 = fx;
            if (lx > x1) x1 = lx;
            if (y < y0) y0 = y;
            y1 = y;
        }
    }
    SlotMeta m{0, 0, 0, 0, 0, 0, 0, 0};
    if (x1 >= 0) { m.x0 = x0 & ~7; m.y0 = y0; m.x1 = std::min(gw, (x1 + 8) & ~7); m.y1 = y1 + 1; }
    if ((uint32_t)(m.x1 - m.x0) > h->geom.pw || (uint32_t)(m.y1 - m.y0) > h->geom.ph)
        return fail(h, SLAMRS_E_WINDOW, "the image's informed extent does not fit the windowed grid slot");
    // dense image -> scratch, then scattered into the slot (whole-grid slots: a plain row copy)
    CU_TRY(h, cudaMemcpyAsync(h->d_export, cells, sizeof(uint32_t) * h->n_cells, cudaMemcpyHostToDevice, h->stream));
    CU_TRY(h, cudaMemsetAsync(h->d_cells + (size_t)slot * h->cells_per_grid, 0, sizeof(uint32_t) * h->cells_per_grid, h->stream));
    launch_import_slot(h->stream, reinterpret_cast<const uint32_t*>(h->d_export), h->d_cells + (size_t)slot * h->cells_per_grid,
                       m, h->geom);
    h->launches++;
    CU_TRY(h, cudaMemcpyAsync(h->d_meta + slot, &m, sizeof(m), cudaMemcpyHostToDevice, h->stream));
    // band extents of the image (0 for every band without informed cells)
    std::vector<uint32_t> bands(h->n_bands, 0u);
    for (int y = 0; y < gh; ++y) {
        const uint32_t* row = cells + (size_t)y * gw;
        int fx = -1, lx = -1;
        for (int x = 0; x < gw; ++x)
            if (row[x]) { if (fx < 0) fx = x; lx = x; }
        if (fx < 0) continue;
        uint32_t& e = bands[phys_band(h->geom, (uint32_t)y)];
        uint32_t bx0 = (uint32_t)fx & ~7u, bx1 = std::min((uint32_t)gw, ((uint32_t)lx + 8u) & ~7u);
        if (e) { bx0 = std::min(bx0, e & 0xffffu); bx1 = std::max(bx1, e >> 16); }
        e = bx0 | (bx1 << 16);
    }
    CU_TRY(h, cudaMemcpyAsync(h->d_bands + (size_t)slot * h->n_bands, bands.data(), sizeof(uint32_t) * h->n_bands,
                              cudaMemcpyHostToDevice, h->stream));
    h->est_box_stale = true;
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    return SLAMRS_OK;
}

int slamrs_gpu_get_extents(slamrs_gpu_handle* h, uint64_t particle, int32_t out_box_shift[5], uint32_t* out_bands,
                           uint32_t* out_n_bands) {
    if (!h || !out_box_shift) return SLAMRS_E_INVALID_ARG;
    if (h->localizer) return fail(h, SLAMRS_E_INVALID_ARG, NO_GRIDS);
    DeviceGuard g(h->device);
    int32_t slot = 0;
    int rc = local_root_slot(h, particle, &slot);
    if (rc) return rc;
    SlotMeta m;
    CU_TRY(h, cudaMemcpyAsync(&m, h->d_meta + slot, sizeof(m), cudaMemcpyDeviceToHost, h->stream));
    if (out_bands)
        CU_TRY(h, cudaMemcpyAsync(out_bands, h->d_bands + (size_t)slot * h->n_bands, sizeof(uint32_t) * h->n_bands,
                                  cudaMemcpyDeviceToHost, h->stream));
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    out_box_shift[0] = m.x0; out_box_shift[1] = m.y0; out_box_shift[2] = m.x1; out_box_shift[3] = m.y1; out_box_shift[4] = 0;
    if (out_n_bands) *out_n_bands = h->n_bands;
    return SLAMRS_OK;
}

int slamrs_gpu_get_log_odds(slamrs_gpu_handle* h, uint64_t particle, double* out_cells) {
    if (!h || !out_cells) return SLAMRS_E_INVALID_ARG;
    if (h->localizer) return fail(h, SLAMRS_E_INVALID_ARG, NO_GRIDS);
    DeviceGuard g(h->device);
    int32_t slot = 0;
    int rc = local_root_slot(h, particle, &slot);
    if (rc) return rc;
    launch_export_slot(h->stream, h->d_cells + (size_t)slot * h->cells_per_grid, h->d_meta + slot, h->geom, true, h->d_export);
    h->launches++;
    CU_TRY(h, cudaMemcpyAsync(out_cells, h->d_export, sizeof(double) * h->n_cells, cudaMemcpyDeviceToHost, h->stream));
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    return SLAMRS_OK;
}

// ------------------------------------------------------------------ kernel-level test hooks

int slamrs_gpu_debug_raycast(int device, const float* x0, const float* y0, const float* x1, const float* y1,
                             uint32_t n_rays, uint32_t grid_w, uint32_t grid_h, uint32_t extra_steps, int32_t* out_xy,
                             uint32_t cap, uint32_t* out_count) {
    if (!x0 || !y0 || !x1 || !y1 || !out_xy || !out_count || n_rays == 0 || cap == 0) return SLAMRS_E_INVALID_ARG;
    int rc = debug_device(device);
    if (rc) return rc;
    DeviceGuard g(device < 0 ? 0 : device);
    DevBuf<float> a, b, c, d;
    DevBuf<int32_t> o;
    DevBuf<uint32_t> cnt;
    DBG_CU(a.alloc(n_rays)); DBG_CU(b.alloc(n_rays)); DBG_CU(c.alloc(n_rays)); DBG_CU(d.alloc(n_rays));
    DBG_CU(o.alloc((size_t)n_rays * cap * 2)); DBG_CU(cnt.alloc(n_rays));
    DBG_CU(cudaMemcpy(a.p, x0, 4 * n_rays, cudaMemcpyHostToDevice));
    DBG_CU(cudaMemcpy(b.p, y0, 4 * n_rays, cudaMemcpyHostToDevice));
    DBG_CU(cudaMemcpy(c.p, x1, 4 * n_rays, cudaMemcpyHostToDevice));
    DBG_CU(cudaMemcpy(d.p, y1, 4 * n_rays, cudaMemcpyHostToDevice));
    DBG_CU(cudaMemset(o.p, 0xff, sizeof(int32_t) * (size_t)n_rays * cap * 2));
    launch_debug_raycast(nullptr, a.p, b.p, c.p, d.p, n_rays, grid_w, grid_h, extra_steps, o.p, cap, cnt.p);
    DBG_CU(cudaGetLastError());
    DBG_CU(cudaMemcpy(out_xy, o.p, sizeof(int32_t) * (size_t)n_rays * cap * 2, cudaMemcpyDeviceToHost));
    DBG_CU(cudaMemcpy(out_count, cnt.p, 4 * n_rays, cudaMemcpyDeviceToHost));
    return SLAMRS_OK;
}

int slamrs_gpu_debug_sincos(int device, const float* x, uint32_t n, float* out_sin, float* out_cos) {
    if (!x || !out_sin || !out_cos || n == 0) return SLAMRS_E_INVALID_ARG;
    int rc = debug_device(device);
    if (rc) return rc;
    DeviceGuard g(device < 0 ? 0 : device);
    DevBuf<float> a, s, c;
    DBG_CU(a.alloc(n)); DBG_CU(s.alloc(n)); DBG_CU(c.alloc(n));
    DBG_CU(cudaMemcpy(a.p, x, 4 * (size_t)n, cudaMemcpyHostToDevice));
    launch_debug_sincos(nullptr, a.p, n, s.p, c.p);
    DBG_CU(cudaGetLastError());
    DBG_CU(cudaMemcpy(out_sin, s.p, 4 * (size_t)n, cudaMemcpyDeviceToHost));
    DBG_CU(cudaMemcpy(out_cos, c.p, 4 * (size_t)n, cudaMemcpyDeviceToHost));
    return SLAMRS_OK;
}

int slamrs_gpu_debug_stream(int device, uint64_t seed, uint64_t step, uint64_t first, uint64_t count, double* out_z,
                            double* out_u) {
    if (!out_u || (count && !out_z)) return SLAMRS_E_INVALID_ARG;
    int rc = debug_device(device);
    if (rc) return rc;
    DeviceGuard g(device < 0 ? 0 : device);
    DevBuf<double> z, u;
    DBG_CU(z.alloc(2 * count)); DBG_CU(u.alloc(1));
    launch_debug_stream(nullptr, seed, step, first, count, z.p, u.p);
    DBG_CU(cudaGetLastError());
    if (count) DBG_CU(cudaMemcpy(out_z, z.p, sizeof(double) * 2 * count, cudaMemcpyDeviceToHost));
    DBG_CU(cudaMemcpy(out_u, u.p, sizeof(double), cudaMemcpyDeviceToHost));
    return SLAMRS_OK;
}

int slamrs_gpu_debug_resample(int device, const double* raw_weights, uint32_t n, double u01, uint32_t* out_idx,
                              uint64_t* out_max_particle, double* out_norm, double* out_cum, uint64_t out_info[4],
                              float out_us[2]) {
    return slamrs_gpu_debug_resample_adaptive(device, raw_weights, n, u01, 0.0, out_idx, out_max_particle, out_norm, out_cum,
                                              out_info, out_us, nullptr, nullptr, nullptr);
}

int slamrs_gpu_debug_resample_adaptive(int device, const double* raw_weights, uint32_t n, double u01, double tau,
                                       uint32_t* out_idx, uint64_t* out_max_particle, double* out_norm, double* out_cum,
                                       uint64_t out_info[4], float out_us[2], double* out_n_eff, uint64_t* out_do_resample,
                                       uint64_t out_shape[4]) {
    if (!raw_weights || !out_idx || n == 0 || n > 0x7fffffffu || !(tau >= 0.0 && tau <= 1.0)) return SLAMRS_E_INVALID_ARG;
    int rc = debug_device(device);
    if (rc) return rc;
    DeviceGuard g(device < 0 ? 0 : device);
    DBG_CU(configure_kernels());
    DevBuf<ParticleResult> res;
    DevBuf<double> wn, cum, fold, u;
    DevBuf<uint32_t> idx;
    DevBuf<StepCounters> cnt;
    DBG_CU(res.alloc(n)); DBG_CU(wn.alloc(n)); DBG_CU(cum.alloc(n)); DBG_CU(fold.alloc(weights_scratch_doubles()));
    DBG_CU(u.alloc(1)); DBG_CU(idx.alloc(n)); DBG_CU(cnt.alloc(1));
    std::vector<ParticleResult> host(n);
    for (uint32_t i = 0; i < n; ++i) { host[i].weight = raw_weights[i]; host[i].x = host[i].y = host[i].theta = 0.0f; host[i].slot = 0; }
    DBG_CU(cudaMemcpy(res.p, host.data(), sizeof(ParticleResult) * (size_t)n, cudaMemcpyHostToDevice));
    DBG_CU(cudaMemcpy(u.p, &u01, sizeof(double), cudaMemcpyHostToDevice));
    DBG_CU(cudaMemset(cnt.p, 0, sizeof(StepCounters)));
    cudaEvent_t ev[3];
    for (auto& e : ev) DBG_CU(cudaEventCreate(&e));
    const int reps = out_us ? 20 : 1;
    float us[2] = {0.f, 0.f};
    for (int r = 0; r < reps; ++r) {
        cudaEventRecord(ev[0], nullptr);
        launch_weights(nullptr, res.p, n, wn.p, cum.p, fold.p, tau, cnt.p);
        cudaEventRecord(ev[1], nullptr);
        launch_resample_indices(nullptr, res.p, cum.p, n, u.p, 0, 0, idx.p, nullptr, 0, 0, false, nullptr,
                                RayLists{nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, 0u, 0u}, wn.p, nullptr, cnt.p);
        cudaEventRecord(ev[2], nullptr);
        cudaError_t e = cudaDeviceSynchronize();
        if (e != cudaSuccess) { for (auto& x : ev) cudaEventDestroy(x); return fail(nullptr, SLAMRS_E_CUDA, cudaGetErrorString(e)); }
        float a = 0.f, b = 0.f;
        cudaEventElapsedTime(&a, ev[0], ev[1]); cudaEventElapsedTime(&b, ev[1], ev[2]);
        if (r > 0 || reps == 1) { us[0] += a * 1000.f; us[1] += b * 1000.f; }
    }
    for (auto& e : ev) cudaEventDestroy(e);
    if (out_us) { out_us[0] = us[0] / (float)(reps > 1 ? reps - 1 : 1); out_us[1] = us[1] / (float)(reps > 1 ? reps - 1 : 1); }
    StepCounters c;
    DBG_CU(cudaMemcpy(&c, cnt.p, sizeof(c), cudaMemcpyDeviceToHost));
    DBG_CU(cudaMemcpy(out_idx, idx.p, sizeof(uint32_t) * (size_t)n, cudaMemcpyDeviceToHost));
    if (out_norm) DBG_CU(cudaMemcpy(out_norm, wn.p, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost));
    if (out_cum) DBG_CU(cudaMemcpy(out_cum, cum.p, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost));
    if (out_max_particle) *out_max_particle = c.max_particle;
    if (out_us && getenv("SLAMRS_FOLD_TRACE_PRINT")) {
        long long tr[64];
        if (weights_trace(tr) == 0) {
            fprintf(stderr, "k_weights clock stamps (cycles from start):");
            for (int k = 0; k < 44; ++k) fprintf(stderr, " [%d]%lld", k, tr[k] ? tr[k] - tr[0] : -1);
            fprintf(stderr, "\n");
        }
    }
    if (out_info) { out_info[0] = c.clamped; out_info[1] = c.fold_rounds; out_info[2] = c.fold_heads; out_info[3] = c.fold_fallback; }
    if (out_n_eff) *out_n_eff = c.n_eff;
    if (out_do_resample) *out_do_resample = c.do_resample;
    if (out_shape) {
        const WeightsShape sh = weights_shape(n);
        out_shape[0] = sh.cluster; out_shape[1] = sh.threads; out_shape[2] = sh.chunk; out_shape[3] = sh.regs ? 1u : 0u;
    }
    return SLAMRS_OK;
}

}  // extern "C"
