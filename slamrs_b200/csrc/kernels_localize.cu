// Monte Carlo localisation against one shared, read-only occupancy map: the per-cell sensor-term table built once
// at create (k_loc_terms_beam, or k_loc_dt_cols + k_loc_dt_rows for the likelihood field) and the per-step kernel
// k_loc_step (motion + likelihood, fused). k_weights and k_resample_indices run unchanged behind it.
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

}  // namespace slamrs
