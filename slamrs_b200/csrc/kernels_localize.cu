// Monte Carlo localisation against one shared, read-only occupancy map: the per-cell sensor-term table built once
// at create (k_loc_terms_beam, or k_loc_dt_cols + k_loc_dt_rows for the likelihood field) and the per-step kernel
// k_loc_step (motion + likelihood, fused). k_weights and k_resample_indices run unchanged behind it, and with
// recovery on (slamrs_gpu_set_recovery) k_loc_recover behind them, on the free-cell list built at create. With
// KLD-sampling on (slamrs_gpu_set_kld) k_loc_kld runs in front of k_loc_step and sizes the next generation.
#include "kernels_common.cuh"

namespace slamrs {

// =============================================================================== term tables
// Beam-endpoint model (the reference's, map.rs:130-141): the factor of the loaded probability, the same expression
// k_likelihood evaluates on the probability k_export produces from the same counters.
__global__ void __launch_bounds__(256) k_loc_terms_beam(const double* __restrict__ prob, size_t n_cells, double* __restrict__ terms) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_cells) terms[i] = beam_log_term_p(prob[i]);
}

// Likelihood field: exact squared Euclidean distance (in cells) to the nearest obstacle, in two separable passes.
constexpr uint32_t DT_NONE = 0xffffffffu;
// Column pass: g[y * w + x] = distance from row y to the nearest obstacle row of column x (DT_NONE: the column has
// none). One thread per column (coalesced across a row), a sweep down and a sweep up.
__global__ void __launch_bounds__(256) k_loc_dt_cols(const double* __restrict__ prob, uint32_t w, double occupied_above,
                                                     uint32_t* __restrict__ g) {
    const uint32_t x = blockIdx.x * blockDim.x + threadIdx.x;
    if (x >= w) return;
    uint32_t last = DT_NONE;
    for (uint32_t y = 0; y < w; ++y) {
        if (prob[(size_t)y * w + x] > occupied_above) last = y;
        g[(size_t)y * w + x] = last == DT_NONE ? DT_NONE : y - last;
    }
    last = DT_NONE;
    for (uint32_t y = w; y-- > 0;) {
        if (prob[(size_t)y * w + x] > occupied_above) last = y;
        if (last != DT_NONE && last - y < g[(size_t)y * w + x]) g[(size_t)y * w + x] = last - y;
    }
}
// Row pass: d2(x, y) = min over x' of (x - x')^2 + g(x', y)^2, searched outward from x until (x - x')^2 alone reaches
// the best value found (every farther x' is at least that far), then the field term
//     log(z_hit * exp(((-0.5 * d2) * res^2) / sigma^2) + z_rand)
// One CTA per row, the row's column distances in shared memory. A map without obstacles (no column has one) gets
// log(z_rand) everywhere.
__global__ void __launch_bounds__(256) k_loc_dt_rows(const uint32_t* __restrict__ g, uint32_t w, double zh, double zr, double rr,
                                                     double ss, double* __restrict__ terms) {
    extern __shared__ uint32_t s_g[];
    const uint32_t y = blockIdx.x;
    int any = 0;
    for (uint32_t x = threadIdx.x; x < w; x += blockDim.x) {
        const uint32_t v = g[(size_t)y * w + x];
        s_g[x] = v;
        any |= v != DT_NONE;
    }
    const bool obstacles = __syncthreads_or(any) != 0;
    for (uint32_t x = threadIdx.x; x < w; x += blockDim.x) {
        double t = log(zr);
        if (obstacles) {
            unsigned long long best = ~0ull;
            for (uint32_t k = 0; k < w; ++k) {
                const unsigned long long k2 = (unsigned long long)k * k;
                if (k2 >= best) break;
                if (k <= x && s_g[x - k] != DT_NONE) best = min(best, k2 + (unsigned long long)s_g[x - k] * s_g[x - k]);
                if (x + k < w && s_g[x + k] != DT_NONE) best = min(best, k2 + (unsigned long long)s_g[x + k] * s_g[x + k]);
            }
            t = log(__dadd_rn(__dmul_rn(zh, exp(__ddiv_rn(__dmul_rn(__dmul_rn(-0.5, (double)best), rr), ss))), zr));
        }
        terms[(size_t)y * w + x] = t;
    }
}

cudaError_t launch_loc_terms(cudaStream_t stream, const double* prob, uint32_t w, int field, float sigma, float z_rand,
                             float occupied_above, float res, uint32_t* scratch, double* terms) {
    const size_t n_cells = (size_t)w * w;
    if (!field) {
        k_loc_terms_beam<<<(unsigned)((n_cells + 255) / 256), 256, 0, stream>>>(prob, n_cells, terms);
        return cudaGetLastError();
    }
    const double zr = (double)z_rand, zh = 1.0 - zr, rr = (double)res * (double)res, ss = (double)sigma * (double)sigma;
    k_loc_dt_cols<<<(w + 255) / 256, 256, 0, stream>>>(prob, w, (double)occupied_above, scratch);
    const size_t smem = sizeof(uint32_t) * w;
    if (smem > 48u * 1024u) {
        const cudaError_t e = cudaFuncSetAttribute(k_loc_dt_rows, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    k_loc_dt_rows<<<w, 256, smem, stream>>>(scratch, w, zh, zr, rr, ss, terms);
    return cudaGetLastError();
}

// =============================================================================== k_loc_step
// One localisation step's motion and likelihood. Each warp takes 32 particles: lane j samples the motion of particle
// j (motion_step, as k_motion does), then the warp walks the 32 particles one by one with its lanes over the valid
// beams, exactly as k_likelihood does: lane l adds the terms of valid beams l, l+32, l+64, ... in increasing order,
// then the xor butterfly 16, 8, 4, 2, 1. With the same term values the raw weights are therefore bitwise equal to the
// SLAM step's. A beam endpoint inside the grid adds term[row * grid_h + column] (one 8-byte gather from the table,
// which stays in L2), one outside the grid adds `outside`.
// The CTA compacts the valid beams of up to LOC_WIN scan beams at a time into shared memory; a scan longer than
// that keeps the lane sums of its particles in dynamic shared memory between the windows.
constexpr int LOC_WARPS = 4;          // block_compact_valid_beams is written for 128 threads
constexpr uint32_t LOC_WIN = 1024;
constexpr int LOC_UNROLL = 4;         // gathers in flight per lane

__global__ void __launch_bounds__(LOC_WARPS * 32)
k_loc_step(MapGeom geom, OdomModel od, ScanDevice scan, const float* __restrict__ pose_cur, ParticleResult* __restrict__ results,
           uint32_t n, const double* __restrict__ z_draws, uint64_t seed, uint64_t step, const double* __restrict__ terms,
           double outside, const double* __restrict__ carry, const StepCounters* __restrict__ counters) {
    __shared__ float2 s_beams[LOC_WIN];
    extern __shared__ double s_acc[];   // scans of more than LOC_WIN beams: [LOC_WARPS][32 particles][32 lanes]
    pdl_launch_dependents();            // (k_weights, one cluster, may become resident; it waits for this grid)
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const uint32_t p0 = (blockIdx.x * LOC_WARPS + (uint32_t)wid) * 32u;
    const uint32_t p = p0 + (uint32_t)lane;
    ParticleResult r{0.0, 0.0f, 0.0f, 0.0f, -1};
    if (p < n) r = motion_step(od, pose_cur, p, p, z_draws, seed, step);
    const uint32_t cnt = p0 < n ? min(32u, n - p0) : 0u;   // warp-uniform
    double* acc = s_acc + (size_t)wid * 32u * 32u;
    double mine = log(1.0);   // lane j: log-likelihood of particle p0 + j
    uint32_t t_base = 0;      // valid beams before the current window
    for (uint32_t w0 = 0; w0 < scan.n_beams; w0 += LOC_WIN) {   // CTA-uniform
        const uint32_t w1 = min(scan.n_beams, w0 + LOC_WIN);
        __syncthreads();   // every warp is done with the previous window's beams
        const uint32_t k = block_compact_valid_beams(scan, w0, w1, s_beams);
        const bool last = w1 == scan.n_beams;
        const uint32_t i0 = ((uint32_t)lane - t_base) & 31u;   // first beam of this window whose valid index is lane (mod 32)
        for (uint32_t j = 0; j < cnt; ++j) {
            const float nx = __shfl_sync(0xffffffffu, r.x, (int)j);
            const float ny = __shfl_sync(0xffffffffu, r.y, (int)j);
            const float nt = __shfl_sync(0xffffffffu, r.theta, (int)j);
            double lp = w0 == 0 ? log(1.0) : acc[j * 32u + (uint32_t)lane];
            for (uint32_t b = i0; b < k; b += 32u * LOC_UNROLL) {
                double term[LOC_UNROLL];
#pragma unroll
                for (int u = 0; u < LOC_UNROLL; ++u) {
                    const uint32_t i = b + 32u * (uint32_t)u;
                    term[u] = outside;
                    if (i < k) {
                        const float2 ad = s_beams[i];
                        float ex, ey;
                        beam_endpoint(nx, ny, nt, ad.x, ad.y, &ex, &ey);
                        const float gx = world_to_grid(ex, geom.pos_x, geom.res);
                        const float gy = world_to_grid(ey, geom.pos_y, geom.res);
                        if (grid_is_valid(gx, gy, geom.gw, geom.gh))
                            term[u] = __ldg(&terms[(size_t)f32_as_usize(gy) * geom.gh + (size_t)f32_as_usize(gx)]);
                    }
                }
#pragma unroll
                for (int u = 0; u < LOC_UNROLL; ++u)
                    if (b + 32u * (uint32_t)u < k) lp = __dadd_rn(lp, term[u]);
            }
            if (last) {
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) lp = __dadd_rn(lp, __shfl_xor_sync(0xffffffffu, lp, o));
                if ((uint32_t)lane == j) mine = lp;
            } else {
                acc[j * 32u + (uint32_t)lane] = lp;
            }
        }
        t_base += k;
    }
    if (p >= n) return;
    // weight.prob().value(), slam.rs:71: exp(log p(z|x,m) + log p(x'|x,u)); adaptive resampling carries the weights of a
    // step that did not resample (as k_likelihood does)
    ParticleResult out = r;
    out.weight = exp(__dadd_rn(mine, r.weight));
    if (carry != nullptr && counters->carry_active) out.weight = __dmul_rn(carry[p], out.weight);
    results[p] = out;
}

void launch_loc_step(cudaStream_t stream, MapGeom geom, OdomModel od, ScanDevice scan, const float* pose_cur,
                     ParticleResult* results, uint32_t n, const double* z_draws, uint64_t seed, uint64_t step,
                     const double* terms, double outside, const double* carry, const StepCounters* counters) {
    const uint32_t per_cta = LOC_WARPS * 32u;
    const size_t smem = scan.n_beams > LOC_WIN ? sizeof(double) * LOC_WARPS * 32u * 32u : 0u;
    k_loc_step<<<(n + per_cta - 1u) / per_cta, per_cta, smem, stream>>>(geom, od, scan, pose_cur, results, n, z_draws, seed,
                                                                         step, terms, outside, carry, counters);
}

// =============================================================================== recovery (augmented MCL)
// Free-cell list at create: an ordered compaction of p < 0.5 over the uploaded map in three launches -- the free cells
// of every tile of FREE_TILE cells (k_loc_free_count), the exclusive scan of those counts (k_loc_free_scan, one CTA)
// and the write of each tile's cells from its offset (k_loc_free_cells). Thread t of a tile owns its cells 8t .. 8t+7.
constexpr uint32_t FREE_THREADS = 1024, FREE_PER_THREAD = 8, FREE_TILE = FREE_THREADS * FREE_PER_THREAD;

__device__ __forceinline__ uint32_t free_bits(const double* __restrict__ prob, size_t n_cells, size_t base) {
    uint32_t bits = 0;
#pragma unroll
    for (uint32_t k = 0; k < FREE_PER_THREAD; ++k)
        if (base + k < n_cells && prob[base + k] < 0.5) bits |= 1u << k;
    return bits;
}

__global__ void __launch_bounds__(FREE_THREADS) k_loc_free_count(const double* __restrict__ prob, size_t n_cells,
                                                                 uint32_t* __restrict__ counts) {
    __shared__ uint32_t s_tot[33];
    const size_t base = (size_t)blockIdx.x * FREE_TILE + (size_t)threadIdx.x * FREE_PER_THREAD;
    uint32_t total;
    block_excl_scan_u32((uint32_t)__popc(free_bits(prob, n_cells, base)), s_tot, &total);
    if (threadIdx.x == 0) counts[blockIdx.x] = total;
}

__global__ void __launch_bounds__(FREE_THREADS) k_loc_free_scan(uint32_t* __restrict__ counts, uint32_t n_tiles) {
    __shared__ uint32_t s_tot[33];
    uint32_t carry = 0;
    for (uint32_t i0 = 0; i0 < n_tiles; i0 += FREE_THREADS) {   // CTA-uniform
        const uint32_t i = i0 + threadIdx.x;
        uint32_t total;
        const uint32_t ex = block_excl_scan_u32(i < n_tiles ? counts[i] : 0u, s_tot, &total);
        if (i < n_tiles) counts[i] = carry + ex;
        carry += total;
    }
}

__global__ void __launch_bounds__(FREE_THREADS) k_loc_free_cells(const double* __restrict__ prob, size_t n_cells,
                                                                 const uint32_t* __restrict__ offsets,
                                                                 uint32_t* __restrict__ free_cells) {
    __shared__ uint32_t s_tot[33];
    const size_t base = (size_t)blockIdx.x * FREE_TILE + (size_t)threadIdx.x * FREE_PER_THREAD;
    uint32_t bits = free_bits(prob, n_cells, base);
    uint32_t total;
    uint32_t o = offsets[blockIdx.x] + block_excl_scan_u32((uint32_t)__popc(bits), s_tot, &total);
    for (; bits; bits &= bits - 1u) free_cells[o++] = (uint32_t)(base + (uint32_t)(__ffs(bits) - 1));
}

size_t loc_free_scratch_words(size_t n_cells) { return (n_cells + FREE_TILE - 1) / FREE_TILE; }

void launch_loc_free_cells(cudaStream_t stream, const double* prob, size_t n_cells, uint32_t* scratch, uint32_t* free_cells) {
    const uint32_t n_tiles = (uint32_t)loc_free_scratch_words(n_cells);
    k_loc_free_count<<<n_tiles, FREE_THREADS, 0, stream>>>(prob, n_cells, scratch);
    k_loc_free_scan<<<1, FREE_THREADS, 0, stream>>>(scratch, n_tiles);
    k_loc_free_cells<<<n_tiles, FREE_THREADS, 0, stream>>>(prob, n_cells, scratch, free_cells);
}

void launch_tile_offsets(cudaStream_t stream, uint32_t* counts, uint32_t n_tiles) {
    k_loc_free_scan<<<1, FREE_THREADS, 0, stream>>>(counts, n_tiles);
}

// One thread per new particle, behind k_resample_indices. Every thread computes the same new state from the previous
// step's (slot (step + 1) & 1); thread 0 stores it in slot step & 1 and clears the other slot's count for the next
// step. With p > 0 a thread draws its particle's decision (slamrs_stream::recovery_draw) and replaces the resampled
// pose; each warp adds its injections to the count with one atomic. The estimate, the indices and the weights that
// k_weights and k_resample_indices recorded stay as they are.
// n particles were weighted (w_avg = sum / n) and m new ones drawn (the injection candidates); m = n unless KLD-sampling
// sized the new generation.
__global__ void __launch_bounds__(256)
k_loc_recover(uint32_t n, uint32_t m_draws, const StepCounters* __restrict__ counters, RecoveryState* state, uint64_t step,
              double alpha_slow, double alpha_fast, uint64_t seed, const uint32_t* __restrict__ free_cells, uint32_t n_free,
              uint32_t grid_h, double pos_x, double pos_y, double res, float* __restrict__ pose_next) {
    pdl_wait();   // k_resample_indices has completed (it waited for k_weights): counters->sum, the resampled poses
    RecoveryState* prev = state + ((step + 1u) & 1u);
    RecoveryState* cur = state + (step & 1u);
    double w_slow = prev->w_slow, w_fast = prev->w_fast;
    const double p = slamrs_stream::recovery_update(counters->sum, n, alpha_slow, alpha_fast, &w_slow, &w_fast);
    const uint32_t m = blockIdx.x * blockDim.x + threadIdx.x;
    if (m == 0) {
        cur->w_slow = w_slow; cur->w_fast = w_fast; cur->p = p;
        prev->injected = 0ull;
    }
    if (!(p > 0.0)) return;   // (grid-uniform)
    float x, y, t;
    const bool inj = m < m_draws && slamrs_stream::recovery_draw(seed, step, m, p, free_cells, n_free, grid_h, pos_x, pos_y, res,
                                                           &x, &y, &t);
    const unsigned mask = __ballot_sync(0xffffffffu, inj);
    if (inj) {
        float* q = pose_next + 3 * (size_t)m;
        q[0] = x; q[1] = y; q[2] = t;
    }
    if ((threadIdx.x & 31u) == 0 && mask) atomicAdd(&cur->injected, (unsigned long long)__popc(mask));
}

void launch_loc_recover(cudaStream_t stream, uint32_t n, uint32_t m_draws, const StepCounters* counters, RecoveryState* state,
                        uint64_t step, double alpha_slow, double alpha_fast, uint64_t seed, const uint32_t* free_cells,
                        uint32_t n_free, MapGeom geom, float* pose_next) {
    launch_pdl(k_loc_recover, dim3((m_draws + 255u) / 256u), dim3(256), 0, stream, n, m_draws, counters, state, step, alpha_slow,
               alpha_fast, seed, free_cells, n_free, geom.gh, (double)geom.pos_x, (double)geom.pos_y, (double)geom.res, pose_next);
}

// =============================================================================== KLD-sampling (adaptive population)
// The particle count of the next generation for k occupied bins: AMCL's pf_resample_limit in its order of operations
// (n_min instead of max_particles for k <= 1).
__device__ __forceinline__ uint32_t kld_bound(uint32_t k, const KldParams& kp) {
    if (k <= 1u) return kp.n_min;
    const double km1 = (double)(k - 1u);
    const double b = __ddiv_rn(2.0, __dmul_rn(9.0, km1));
    const double x = __dadd_rn(__dsub_rn(1.0, b), __dmul_rn(__dsqrt_rn(b), kp.z));
    const double n = __dmul_rn(__dmul_rn(__dmul_rn(__ddiv_rn(km1, __dmul_rn(2.0, kp.err)), x), x), x);
    if (!(n < (double)kp.n_max)) return kp.n_max;   // (also NaN and infinity)
    const double c = ceil(n);
    return c < (double)kp.n_min ? kp.n_min : (uint32_t)c;
}

// One thread per pose of the starting generation: marks its bin in the bitmap (state + KLD_HEADER_WORDS, zeroed with the
// header before the launch) and each warp adds the bits it set first to state[0]. The last CTA to finish (ticket
// state[1]) evaluates the bound and leaves {n, k, N_next} in the host's page-locked result. A converged cloud puts
// nearly every pose into a few bins: only one lane per distinct bin of a warp touches the bitmap, and it reads the word
// before its atomicOr, so only the first warps to reach a bin contend for that word.
__global__ void __launch_bounds__(256)
k_loc_kld(const float* __restrict__ pose, uint32_t n, MapGeom geom, KldParams kp, uint32_t* state, KldResult* host_out) {
    __shared__ bool s_last;
    uint32_t* bits = state + KLD_HEADER_WORDS;
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t b = 0xffffffffu;   // (no bin: bins stay below 2^28)
    if (i < n) {
        const float* q = pose + 3 * (size_t)i;
        b = kld_bin(q[0], q[1], q[2], geom, kp);
    }
    const unsigned peers = __match_any_sync(0xffffffffu, b);
    bool fresh = false;
    if (i < n && (threadIdx.x & 31u) == (unsigned)(__ffs(peers) - 1)) {
        const uint32_t bit = 1u << (b & 31u);
        uint32_t* w = &bits[b >> 5];
        if ((*(volatile const uint32_t*)w & bit) == 0u) fresh = (atomicOr(w, bit) & bit) == 0u;
    }
    const unsigned mask = __ballot_sync(0xffffffffu, fresh);
    if ((threadIdx.x & 31u) == 0 && mask) atomicAdd(&state[0], (uint32_t)__popc(mask));
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = atomicAdd(&state[1], 1u) == gridDim.x - 1u;
    __syncthreads();
    if (!s_last || threadIdx.x != 0) return;
    __threadfence();
    const uint32_t k = atomicAdd(&state[0], 0u);
    host_out->n_weighted = n;
    host_out->k = k;
    host_out->m = kld_bound(k, kp);
    __threadfence_system();
}

void launch_loc_kld(cudaStream_t stream, const float* pose, uint32_t n, MapGeom geom, const KldParams& kp, uint32_t* state,
                    KldResult* host_out) {
    k_loc_kld<<<(n + 255u) / 256u, 256, 0, stream>>>(pose, n, geom, kp, state, host_out);
}

}  // namespace slamrs
