// k_motion (robot.rs:152-183) and k_likelihood (map.rs:113-145), with the multi-GPU exchange fused
// into the likelihood kernel and the peer-flag barrier that completes it.
#include "kernels_common.cuh"

namespace slamrs {

// =============================================================================== k_motion + k_likelihood
// k_motion: one THREAD per particle. Odometry::sample (robot.rs:170-183) and the motion log-density
// Odometry::probabiliy_of (robot.rs:152-167) (motion_step) need a few hundred scalar f64 operations per
// particle and nothing else; giving them a warp or a CTA would multiply the issued instructions by 32.
// The log-density is parked in ParticleResult::weight until k_likelihood folds it in.
__global__ void __launch_bounds__(128)
k_motion(OdomModel od, const float* __restrict__ pose_cur, const int32_t* __restrict__ slot_of,
         ParticleResult* __restrict__ results, uint32_t first_particle, uint32_t n_local,
         const double* __restrict__ z_draws, uint64_t seed, uint64_t step, ScanDevice scan,
         float2* __restrict__ valid_beams, uint32_t* __restrict__ n_valid, uint32_t* __restrict__ zero_words, uint32_t n_zero) {
    pdl_launch_dependents();   // k_likelihood may take its place on the SMs now; it waits for this grid before it reads
    // the ray update's per-step flags and counters start from zero (instead of a memset in front of the step)
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n_zero; i += gridDim.x * blockDim.x) zero_words[i] = 0u;
    // Block 0 also compacts the scan's VALID beams, in beam order, for k_likelihood (the likelihood kernel
    // spent most of its stall cycles on the dependent valid[] -> angle[], dist[] loads)
    if (blockIdx.x == 0) {
        const uint32_t nv = block_compact_valid_beams(scan, 0u, scan.n_beams, valid_beams);
        if (threadIdx.x == 0) *n_valid = nv;
    }
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_local) return;
    const uint32_t gp = first_particle + p;      // global logical index
    ParticleResult r = motion_step(od, pose_cur, p, gp, z_draws, seed, step);
    r.slot = slot_of[p];                    // physical slot, read by other ranks' planners
    results[gp] = r;
}

// k_likelihood: one WARP per particle, lanes over beams. Map::probability_of (map.rs:113-145): one
// gather per valid beam from the PRE-update grid (lanes step through the compacted list of valid
// beams, so every lane of every batch has work). LK_UNROLL gathers are in flight per lane before
// the first exp/log. A never-informed cell (counters 0 -> log-odds 0 -> p = 0.5) contributes
// log(1/1) = 0 and skips the transcendental work. Each lane adds its terms in beam order, the 32
// lane sums are combined by a fixed butterfly: deterministic, order-independent of scheduling.
constexpr int LK_WARPS = 4;
constexpr int LK_UNROLL = 4;

__global__ void __launch_bounds__(LK_WARPS * 32, 2048 / (LK_WARPS * 32))   // every particle of an 8,192-shard resident at once
k_likelihood(MapGeom geom, ScanDevice scan, const int32_t* __restrict__ alias_of, const uint32_t* __restrict__ cells,
             const SlotMeta* __restrict__ meta,
             size_t cells_per_grid, ParticleResult* __restrict__ results, uint32_t first_particle, uint32_t n_local,
             const double* __restrict__ term_table, const float2* __restrict__ valid_beams,
             const uint32_t* __restrict__ n_valid_ptr, const double* __restrict__ carry, const StepCounters* __restrict__ counters,
             ParticleResult* const* __restrict__ peer_results, uint32_t peer_offset, uint32_t rank, uint32_t world) {
    pdl_launch_dependents();   // (k_weights, one CTA, may become resident)
    pdl_wait();                // k_motion has completed: poses, motion log-densities, the compacted beam list
    const uint32_t p = blockIdx.x * LK_WARPS + (threadIdx.x >> 5);
    if (p >= n_local) return;
    const int lane = threadIdx.x & 31;
    const ParticleResult r = results[first_particle + p];
    const float nx = r.x, ny = r.y, ntheta = r.theta;
    // a clone that has not been written since resampling shares its source's cells (PlanArgs::alias_of)
    const int32_t root = alias_of ? alias_of[r.slot] : r.slot;
    const uint32_t* grid = cells + (size_t)root * cells_per_grid;
    const SlotMeta sm = meta[root];      // informed extent (outside it a windowed slot must not be read)

    double lp = log(1.0);
    const uint32_t n_valid = *n_valid_ptr;   // valid beams only, compacted by k_motion (ascending beam index)
    for (uint32_t base = 0; base < n_valid; base += 32u * LK_UNROLL) {
        uint32_t cell[LK_UNROLL];
#pragma unroll
        for (int u = 0; u < LK_UNROLL; ++u) {
            const uint32_t t = base + (uint32_t)u * 32u + (uint32_t)lane;
            cell[u] = 0u;
            if (t < n_valid) {
                const float2 ad = __ldg(&valid_beams[t]);   // (angle, distance) of the t-th valid beam
                float ex, ey;
                beam_endpoint(nx, ny, ntheta, ad.x, ad.y, &ex, &ey);
                const float gx = world_to_grid(ex, geom.pos_x, geom.res);
                const float gy = world_to_grid(ey, geom.pos_y, geom.res);
                if (grid_is_valid(gx, gy, geom.gw, geom.gh)) {
                    const size_t column = (size_t)f32_as_usize(gx), row = (size_t)f32_as_usize(gy);
                    // index(): map.rs:201-204, then the slot's layout
                    if (!geom.windowed || ((int)column >= sm.x0 && (int)column < sm.x1 && (int)row >= sm.y0 && (int)row < sm.y1))
                        cell[u] = __ldg(&grid[phys_index(geom, (uint32_t)column, (uint32_t)row)]);
                }
            }
        }
#pragma unroll
        for (int u = 0; u < LK_UNROLL; ++u) {
            if (cell[u] != 0u) {
                const uint32_t nf = cell[u] & 0xffffu, no = cell[u] >> 16;
                const double term = (nf < LK_TABLE_NF && no < LK_TABLE_NO) ? __ldg(&term_table[nf * LK_TABLE_NO + no])
                                                                           : beam_log_term(cell[u]);
                lp = __dadd_rn(lp, term);
            }
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) lp = __dadd_rn(lp, __shfl_xor_sync(0xffffffffu, lp, o));
    // weight.prob().value(), slam.rs:71: exp(log p(z|x,m) + log p(x'|x,u))
    ParticleResult out = r;
    out.weight = exp(__dadd_rn(lp, r.weight));
    // adaptive resampling (not in the reference): a step that did not resample carries its weights forward
    if (carry != nullptr && counters->carry_active) out.weight = __dmul_rn(carry[first_particle + p], out.weight);
    if (lane == 0) results[first_particle + p] = out;
    // The exchange step, fused: lane q stores the finished record straight into GPU q's copy of
    // the population array over NVLink (24 bytes per particle and peer), so that after one
    // peer barrier every GPU holds every particle's weight, pose and slot.
    if (peer_results != nullptr && (uint32_t)lane < world && (uint32_t)lane != rank)
        peer_results[lane][peer_offset + first_particle + p] = out;
}

void launch_motion_likelihood(cudaStream_t stream, MapGeom geom, OdomModel od, ScanDevice scan,
                              const float* pose_cur, const int32_t* slot_of, const int32_t* alias_of,
                              const uint32_t* cells,
                              const SlotMeta* meta, size_t cells_per_grid, ParticleResult* results, uint32_t first_particle,
                              uint32_t n_local, const double* z_draws, uint64_t seed, uint64_t step,
                              const double* term_table, float2* valid_beams, uint32_t* n_valid,
                              const double* carry, const StepCounters* counters,
                              ParticleResult* const* peer_results, uint32_t peer_offset, uint32_t rank, uint32_t world,
                              uint32_t* zero_words, uint32_t n_zero, const ScanMatchParams* match, uint2* match_stats) {
    k_motion<<<(n_local + 127u) / 128u, 128, 0, stream>>>(od, pose_cur, slot_of, results, first_particle, n_local,
                                                         z_draws, seed, step, scan, valid_beams, n_valid, zero_words, n_zero);
    if (match)   // refines the sampled poses in results[] before the likelihood reads them
        launch_scan_match(stream, geom, *match, od, pose_cur, alias_of, cells, meta, cells_per_grid, results, first_particle,
                          n_local, valid_beams, n_valid, match_stats);
    launch_pdl(k_likelihood, dim3((n_local + LK_WARPS - 1) / LK_WARPS), dim3(LK_WARPS * 32), 0, stream, geom, scan, alias_of, cells,
               meta, cells_per_grid, results, first_particle, n_local, term_table, valid_beams, n_valid, carry, counters,
               peer_results, peer_offset, rank, world);
}

__global__ void k_fill_term_table(double* __restrict__ table) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= LK_TABLE_NF * LK_TABLE_NO) return;
    const uint32_t nf = i / LK_TABLE_NO, no = i % LK_TABLE_NO;
    table[i] = (nf | no) ? beam_log_term(nf | (no << 16)) : 0.0;   // entry (0,0) is never read (prior cells are skipped)
}
void launch_fill_term_table(cudaStream_t stream, double* table) {
    k_fill_term_table<<<(LK_TABLE_NF * LK_TABLE_NO + 255) / 256, 256, 0, stream>>>(table);
}

// =============================================================================== k_peer_barrier
// Stream-ordered barrier across the GPUs of one box through peer-mapped flags: lane q publishes
// this rank's epoch into GPU q's flag array (release, system scope: every write this GPU issued
// before, including the peer stores of earlier kernels in the stream, is visible first) and then
// waits until GPU q's epoch has arrived here (acquire). Epochs only grow, so flags are never reset.
// A bounded wait (timeout_ns, one minute by default: ranks are driven by independent host threads
// that may lag) turns a lost peer into an error instead of a hung GPU.
// Leaving: a rank that destroys its handle publishes PEER_GOODBYE instead of an epoch and waits for
// the same from every peer before it frees the memory they have mapped. A peer that meets the
// goodbye at one of its own barriers is poisoned (barrier_timeout = 2): its step fails at the next
// sync, its owner destroys it, and only then does the first rank free its pool -- a rank that fails
// alone (SLAMRS_E_STAGING, SLAMRS_E_WINDOW) never pulls memory from under kernels its peers have
// already queued.
constexpr unsigned long long PEER_GOODBYE = ~0ull;
__global__ void __launch_bounds__(64)
k_peer_barrier(unsigned long long* const* __restrict__ peer_flags, unsigned long long* my_flags, uint32_t rank,
               uint32_t world, unsigned long long epoch, unsigned long long timeout_ns, StepCounters* counters) {
    pdl_launch_dependents();   // (k_weights may become resident; it waits for this grid)
    pdl_wait();                // the kernel in front (k_likelihood and its peer stores) has completed
    const uint32_t q = threadIdx.x;
    if (q >= world) return;
    const bool leaving = epoch == PEER_GOODBYE;
    __threadfence_system();
    // a flag array holds PEER_MAX_WORLD epochs, then PEER_MAX_WORLD goodbye words (0 until the peer leaves)
    unsigned long long* theirs = peer_flags[q] + rank + (leaving ? PEER_MAX_WORLD : 0u);
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(theirs), "l"(epoch) : "memory");
    // once a barrier has given up the handle is poisoned (the error is reported at the next sync):
    // later barriers publish their epoch, so that healthy peers keep going, but do not wait again
    if (*reinterpret_cast<volatile unsigned long long*>(&counters->barrier_timeout) != 0ull) return;
    const unsigned long long* mine = my_flags + q;
    unsigned long long t0, now, seen = 0ull;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    for (;;) {
        if (!leaving) {
            asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(seen) : "l"(mine) : "memory");
            if (seen >= epoch) break;
        }
        asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(seen) : "l"(mine + PEER_MAX_WORLD) : "memory");
        if (seen == PEER_GOODBYE) {
            if (!leaving) counters->barrier_timeout = 2ull;   // the peer is going away without reaching this barrier
            break;
        }
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
        if (now - t0 > timeout_ns) { counters->barrier_timeout = 1ull; break; }
        __nanosleep(200);
    }
    __threadfence_system();
}

void launch_peer_barrier(cudaStream_t stream, unsigned long long* const* peer_flags, unsigned long long* my_flags,
                         uint32_t rank, uint32_t world, unsigned long long epoch, unsigned long long timeout_ns,
                         StepCounters* counters) {
    launch_pdl(k_peer_barrier, dim3(1), dim3(64), 0, stream, peer_flags, my_flags, rank, world, epoch, timeout_ns, counters);
}
void launch_peer_goodbye(cudaStream_t stream, unsigned long long* const* peer_flags, unsigned long long* my_flags,
                         uint32_t rank, uint32_t world, unsigned long long timeout_ns, StepCounters* counters) {
    k_peer_barrier<<<1, 64, 0, stream>>>(peer_flags, my_flags, rank, world, PEER_GOODBYE, timeout_ns, counters);
}

}  // namespace slamrs
