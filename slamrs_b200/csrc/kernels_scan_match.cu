// k_scan_match: scan-matching pose refinement (not in the reference; the slam.rs:60 TODO). Runs between k_motion and
// k_likelihood when the matcher is on and moves each sampled pose onto its particle's own pre-update grid by a hill
// climb on an integer score (see slamrs_gpu.h and DESIGN.md). The score is a sum of small integers, so its value does
// not depend on the order of the additions and the climb is bit-exact against the CPU oracle.
#include "kernels_common.cuh"

namespace slamrs {

// One WARP per particle, lanes over the compacted valid beams; __reduce_add_sync gives every lane the same total, so
// the climb's decisions are warp-uniform. A round scores all six candidates in one pass over the beams: the four
// translated candidates keep the heading, so they share the current pose's sincos and fl(cs * dist), fl(sn * dist)
// (beam_endpoint is px + fl(cs * dist): bitwise the same endpoints); only the two turned candidates need a sincos each.
constexpr int SM_WARPS = 4;

// [-2, 2]^2 by increasing dx^2 + dy^2; the first (2r + 1)^2 entries are the square of radius r. A beam's score is
// (r+1)^2 - d^2 of the first occupied cell in this order.
__device__ __forceinline__ int match_off_x(int k) {
    constexpr int8_t X[25] = {0, 1, -1, 0, 0, 1, -1, 1, -1, 2, -2, 0, 0, 1, -1, 1, -1, 2, -2, 2, -2, 2, -2, 2, -2};
    return X[k];
}
__device__ __forceinline__ int match_off_y(int k) {
    constexpr int8_t Y[25] = {0, 0, 0, 1, -1, 1, 1, -1, -1, 0, 0, 2, -2, 2, 2, -2, -2, 1, 1, -1, -1, 2, 2, -2, -2};
    return Y[k];
}

struct MatchGrid {
    MapGeom geom;
    const uint32_t* grid;   // the particle's root slot
    SlotMeta sm;            // its informed extent (outside it a windowed slot is the prior and is not read)
    int n_off, rp1sq;       // (2r+1)^2 offsets, (r+1)^2
};

__device__ __forceinline__ uint32_t match_beam_score(const MatchGrid& m, float ex, float ey) {
    const MapGeom& g = m.geom;
    const float gx = world_to_grid(ex, g.pos_x, g.res);
    const float gy = world_to_grid(ey, g.pos_y, g.res);
    if (!grid_is_valid(gx, gy, g.gw, g.gh)) return 0u;
    const uint32_t cx = (uint32_t)f32_as_usize(gx), cy = (uint32_t)f32_as_usize(gy);   // < gw, gh <= 2^31
#pragma unroll
    for (int k = 0; k < 25; ++k) {
        if (k >= m.n_off) break;
        // a negative coordinate wraps to >= 2^32 - 2 > gw, gh
        const uint32_t x = cx + (uint32_t)match_off_x(k), y = cy + (uint32_t)match_off_y(k);
        if (x >= g.gw || y >= g.gh) continue;
        if (g.windowed && !((int)x >= m.sm.x0 && (int)x < m.sm.x1 && (int)y >= m.sm.y0 && (int)y < m.sm.y1)) continue;
        if (cell_occupied(__ldg(&m.grid[phys_index(g, x, y)])))
            return (uint32_t)(m.rp1sq - (match_off_x(k) * match_off_x(k) + match_off_y(k) * match_off_y(k)));
    }
    return 0u;
}

__global__ void __launch_bounds__(SM_WARPS * 32)
k_scan_match(MapGeom geom, ScanMatchParams mp, OdomModel od, const float* __restrict__ pose_cur,
             const int32_t* __restrict__ alias_of, const uint32_t* __restrict__ cells, const SlotMeta* __restrict__ meta,
             size_t cells_per_grid, ParticleResult* __restrict__ results, uint32_t first_particle, uint32_t n_local,
             const float2* __restrict__ valid_beams, const uint32_t* __restrict__ n_valid_ptr, uint2* __restrict__ stats) {
    pdl_wait();   // k_motion has completed: sampled poses, motion log-densities, the compacted beam list
    const uint32_t p = blockIdx.x * SM_WARPS + (threadIdx.x >> 5);
    if (p >= n_local) return;
    const uint32_t lane = threadIdx.x & 31u;
    ParticleResult r = results[first_particle + p];
    const int32_t root = alias_of ? alias_of[r.slot] : r.slot;
    MatchGrid m;
    m.geom = geom;
    m.grid = cells + (size_t)root * cells_per_grid;
    m.sm = meta[root];
    m.n_off = (2 * (int)mp.radius + 1) * (2 * (int)mp.radius + 1);
    m.rp1sq = ((int)mp.radius + 1) * ((int)mp.radius + 1);
    const uint32_t n_valid = *n_valid_ptr;

    float x = r.x, y = r.y, th = r.theta;
    uint32_t s0 = 0u;
    for (uint32_t t = lane; t < n_valid; t += 32u) {
        const float2 ad = __ldg(&valid_beams[t]);
        float ex, ey;
        beam_endpoint(x, y, th, ad.x, ad.y, &ex, &ey);
        s0 += match_beam_score(m, ex, ey);
    }
    uint32_t best = __reduce_add_sync(0xffffffffu, s0);
    uint32_t moves = 0u, scored = 1u;
    for (uint32_t level = 0; level < mp.levels; ++level) {
        const float scale = __int_as_float((127 - (int)level) << 23);   // 2^-level, exact
        const float dxy = __fmul_rn(mp.step_xy, scale), dth = __fmul_rn(mp.step_theta, scale);
        while (moves < mp.max_moves) {
            const float xp = __fadd_rn(x, dxy), xm = __fsub_rn(x, dxy);
            const float yp = __fadd_rn(y, dxy), ym = __fsub_rn(y, dxy);
            const float tp = __fadd_rn(th, dth), tm = __fsub_rn(th, dth);
            uint32_t s[6] = {0u, 0u, 0u, 0u, 0u, 0u};
            for (uint32_t t = lane; t < n_valid; t += 32u) {
                const float2 ad = __ldg(&valid_beams[t]);
                float sn, cs;
                slamrs_libm::sincosf_exact(__fadd_rn(th, ad.x), &sn, &cs);
                const float ox = __fmul_rn(cs, ad.y), oy = __fmul_rn(sn, ad.y);
                s[0] += match_beam_score(m, __fadd_rn(xp, ox), __fadd_rn(y, oy));
                s[1] += match_beam_score(m, __fadd_rn(xm, ox), __fadd_rn(y, oy));
                s[2] += match_beam_score(m, __fadd_rn(x, ox), __fadd_rn(yp, oy));
                s[3] += match_beam_score(m, __fadd_rn(x, ox), __fadd_rn(ym, oy));
                float ex, ey;
                beam_endpoint(x, y, tp, ad.x, ad.y, &ex, &ey);
                s[4] += match_beam_score(m, ex, ey);
                beam_endpoint(x, y, tm, ad.x, ad.y, &ex, &ey);
                s[5] += match_beam_score(m, ex, ey);
            }
            scored += 6u;
            // the first candidate with the largest score
            uint32_t top = __reduce_add_sync(0xffffffffu, s[0]);
            int arg = 0;
#pragma unroll
            for (int k = 1; k < 6; ++k) {
                const uint32_t v = __reduce_add_sync(0xffffffffu, s[k]);
                if (v > top) { top = v; arg = k; }
            }
            if (top <= best) break;
            best = top;
            moves += 1u;
            if (arg == 0) x = xp; else if (arg == 1) x = xm; else if (arg == 2) y = yp;
            else if (arg == 3) y = ym; else if (arg == 4) th = tp; else th = tm;
        }
    }
    if (lane != 0u) return;
    if (moves > 0u) {
        // the motion log-density of the refined pose, from the old pose as k_motion computed it for the sample
        r.weight = motion_log_density(od, pose_cur[3 * p], pose_cur[3 * p + 1], pose_cur[3 * p + 2], x, y, th);
        r.x = x; r.y = y; r.theta = th;
        results[first_particle + p] = r;
    }
    stats[p] = make_uint2(moves, scored);
}

void launch_scan_match(cudaStream_t stream, MapGeom geom, ScanMatchParams mp, OdomModel od, const float* pose_cur,
                       const int32_t* alias_of, const uint32_t* cells, const SlotMeta* meta, size_t cells_per_grid,
                       ParticleResult* results, uint32_t first_particle, uint32_t n_local, const float2* valid_beams,
                       const uint32_t* n_valid, uint2* stats) {
    launch_pdl(k_scan_match, dim3((n_local + SM_WARPS - 1) / SM_WARPS), dim3(SM_WARPS * 32), 0, stream, geom, mp, od,
               pose_cur, alias_of, cells, meta, cells_per_grid, results, first_particle, n_local, valid_beams, n_valid,
               stats);
}

}  // namespace slamrs
