// The ray update: Map::integrate (map.rs:71-106) with GridRayIterator (ray.rs:21-110) and the inverse
// sensor model (map.rs:148-172); hit counters accumulated in a shared-memory disc window, then added to the
// grid. k_ray_update: 32-bit window cells, one CTA per particle (any beam count and grid side).
// k_ray_update_packed / k_ray_update_half: 16-bit window cells and one walk (ray_walk_packed); a whole
// particle per work item written back in place (row-major or windowed slots), or half a particle per work
// item whose write-back also makes a clone's grid private (whole-grid tiled slots).
#include "kernels_common.cuh"
#include <cstdio>
#include <cstdlib>
#include <string>
#include <vector>

namespace slamrs {

// =============================================================================== k_ray_update

constexpr int RAY_MAX_SMEM = 220 * 1024;  // window budget; the HW limit is 227 KB per CTA

// saturating packed add straight to global memory, for the (rare) cells outside the window
__device__ __forceinline__ void global_cell_add(uint32_t* addr, uint32_t inc, bool* saturated) {
    uint32_t old = *addr;
    for (;;) {
        const uint32_t nv = cell_sat_add(old, inc, saturated);
        if (nv == old) return;
        const uint32_t seen = atomicCAS(addr, old, nv);
        if (seen == old) return;
        old = seen;
    }
}

constexpr int RAY_MAX_THREADS = 512;

// touched-extent bookkeeping of one CTA: s_ext = {xmin, ymin, xmax, ymax} (inclusive cells)
__device__ __forceinline__ void ext_init(int* s_ext) {
    if (threadIdx.x == 0) { s_ext[0] = 0x7fffffff; s_ext[1] = 0x7fffffff; s_ext[2] = -1; s_ext[3] = -1; }
}
__device__ __forceinline__ void ext_add(int* s_ext, int xmin, int ymin, int xmax, int ymax) {
    if (xmax < xmin) return;
    atomicMin(&s_ext[0], xmin); atomicMin(&s_ext[1], ymin);
    atomicMax(&s_ext[2], xmax); atomicMax(&s_ext[3], ymax);
}
// union the CTA's touched extent into the slot's box (x aligned to 8 cells); one thread, after a barrier
constexpr int BOX_ALIGN = 8;   // x alignment of extents in cells: one 256-bit access
// Windowed slots: would the informed extent still fit the slot after this scan? `reach` bounds how far
// from the start cell a ray can write (measured range in cells + the slack the host adds). The test is
// conservative (bounding square of the reach) and uniform over the CTA.
__device__ __forceinline__ bool window_would_overflow(const MapGeom& geom, const SlotMeta* meta, int cx0, int cy0, int reach) {
    if (!geom.windowed) return false;
    const SlotMeta m = *meta;
    int x0 = max(0, cx0 - reach) & ~7, x1 = min((int)geom.gw, (min((int)geom.gw, cx0 + reach + 1) + 7) & ~7);
    int y0 = max(0, cy0 - reach), y1 = min((int)geom.gh, cy0 + reach + 1);
    if (m.x1 > m.x0 && m.y1 > m.y0) { x0 = min(x0, m.x0); x1 = max(x1, m.x1); y0 = min(y0, m.y0); y1 = max(y1, m.y1); }
    return (uint32_t)(x1 - x0) > geom.pw || (uint32_t)(y1 - y0) > geom.ph;
}

__device__ __forceinline__ void ext_commit(const int* s_ext, SlotMeta* meta, int gw) {
    if (s_ext[2] < s_ext[0]) return;
    SlotMeta b = *meta;
    const int am = BOX_ALIGN - 1;
    const int x0 = s_ext[0] & ~am, x1 = min(gw, (s_ext[2] + 1 + am) & ~am), y0 = s_ext[1], y1 = s_ext[3] + 1;
    if (b.x1 <= b.x0) { b.x0 = x0; b.y0 = y0; b.x1 = x1; b.y1 = y1; }
    else { b.x0 = min(b.x0, x0); b.y0 = min(b.y0, y0); b.x1 = max(b.x1, x1); b.y1 = max(b.y1, y1); }
    *meta = b;
}
// Band extents of the cells a CTA touches (slam_device.cuh): shared arrays indexed by the band of the
// window row, merged into the slot's band table by band_commit.
constexpr int RAY_MAX_BANDS = (2 * 150 + 1) / BAND_ROWS + 2;
__device__ __forceinline__ void band_init(int* s_blo, int* s_bhi) {
    for (int i = threadIdx.x; i < RAY_MAX_BANDS; i += blockDim.x) { s_blo[i] = 0x7fffffff; s_bhi[i] = -1; }
}
// x range [xlo, xhi] (cells, inclusive) touched in row y; band0 = band of the window's first row
__device__ __forceinline__ void band_add(int* s_blo, int* s_bhi, int band0, int y, int xlo, int xhi) {
    const int lb = y / BAND_ROWS - band0;
    if ((unsigned)lb < (unsigned)RAY_MAX_BANDS) { atomicMin(&s_blo[lb], xlo); atomicMax(&s_bhi[lb], xhi); }
}
// after a barrier: union into the slot's table (8-aligned columns). Rows outside the window's bands
// (cells written through the global path far from the start) fall back to widening by their own band:
// band_add ignores them, so the caller adds them with band_add_global below.
__device__ __forceinline__ void band_commit(const int* s_blo, const int* s_bhi, int band0, uint32_t* bands,
                                            const MapGeom& geom) {
    for (int lb = threadIdx.x; lb < RAY_MAX_BANDS; lb += blockDim.x) {
        if (s_bhi[lb] < s_blo[lb]) continue;
        const uint32_t y = (uint32_t)(band0 + lb) * BAND_ROWS;
        if (y >= geom.gh) continue;
        uint32_t* e = &bands[phys_band(geom, y)];
        const uint32_t old = *e;
        uint32_t x0 = (uint32_t)s_blo[lb] & ~7u, x1 = min(geom.gw, ((uint32_t)s_bhi[lb] + 8u) & ~7u);
        if (old != 0u) { x0 = min(x0, old & 0xffffu); x1 = max(x1, old >> 16); }
        *e = x0 | (x1 << 16);
    }
}
// a single cell written outside the window's bands: widen its band directly (rare, exact path)
__device__ __forceinline__ void band_add_global(uint32_t* bands, const MapGeom& geom, int band0, int x, int y) {
    const int lb = y / BAND_ROWS - band0;
    if ((unsigned)lb < (unsigned)RAY_MAX_BANDS) return;   // covered by the shared arrays
    uint32_t* e = &bands[phys_band(geom, (uint32_t)y)];
    const uint32_t x0n = (uint32_t)x & ~7u, x1n = min(geom.gw, ((uint32_t)x + 8u) & ~7u);
    uint32_t old = *e;
    for (;;) {
        const uint32_t x0 = old ? min(x0n, old & 0xffffu) : x0n, x1 = old ? max(x1n, old >> 16) : x1n;
        const uint32_t nv = x0 | (x1 << 16);
        if (nv == old) return;
        const uint32_t seen = atomicCAS(e, old, nv);
        if (seen == old) return;
        old = seen;
    }
}

constexpr int RAY_MAX_RADIUS = 150;                    // rows of the window: 2 * radius + 1
constexpr int RAY_MAX_ROWS = 2 * RAY_MAX_RADIUS + 1;
constexpr int RAY_WB_BATCH = 6;                        // write-back: global loads in flight per thread

// exact integer square root of a small non-negative integer (same code on host and device so
// that the host's shared-memory sizing and the kernel's row table agree)
__host__ __device__ inline int isqrt_small(int v) {
    int r = (int)sqrtf((float)v);
    while (r * r > v) r--;
    while ((r + 1) * (r + 1) <= v) r++;
    return r;
}

// The window is a DISC of cells around the start cell (rays cannot leave it), stored row by row:
// row dy holds x in [cx - hw, cx + hw], hw = floor(sqrt(R^2 - dy^2)), widened to multiples of 4
// cells for 128-bit write-back. A disc needs pi/4 of the bounding square, which is what lets a
// 6 m range at 5 cm cells (radius 124) fit in one CTA's shared memory.
__host__ __device__ inline int ray_window_cells_upper_bound(int radius, bool vec) {
    int total = 0;
    for (int dy = -radius; dy <= radius; ++dy) total += 2 * isqrt_small(radius * radius - dy * dy) + 1 + (vec ? 6 : 0);
    return total;
}

// A zero-length ray (dx = dy = 0: the endpoint rounds back onto the start point) cannot move, so it emits its start cell
// 1 + additional_steps = 3 times (ray.rs:96-104 with both increments 0). Every other ray emits a cell at most once,
// which is what bounds the window's counters (n_beams hits per cell and scan), so these hits take the exact,
// saturating path instead: a thread tallies them during its walk and sends them after it (at most 3 parked entries
// per ray, within RAY_SPILL_CAP). Every ray of a particle starts in the same cell.
struct ZeroLengthHits {
    uint32_t free_hits = 0u, occ_hits = 0u;
    __device__ __forceinline__ void tally(const RayClassifier& cls, float acc) {
        const uint32_t inc = classify_cell(cls, acc);
        free_hits += inc == CELL_FREE_INC ? 3u : 0u;
        occ_hits += inc == CELL_OCC_INC ? 3u : 0u;
    }
    // returns the hits sent to the exact path
    template <class ExactAdd>
    __device__ __forceinline__ uint32_t flush(int cx0, int cy0, ExactAdd& exact_add, int* s_ext, int* s_blo, int* s_bhi,
                                              int band0) const {
        if (free_hits + occ_hits == 0u) return 0u;
        for (uint32_t k = 0; k < free_hits; ++k) exact_add(cx0, cy0, CELL_FREE_INC);
        for (uint32_t k = 0; k < occ_hits; ++k) exact_add(cx0, cy0, CELL_OCC_INC);
        ext_add(s_ext, cx0, cy0, cx0, cy0);
        band_add(s_blo, s_bhi, band0, cy0, cx0, cx0);
        return free_hits + occ_hits;
    }
};

template <bool kVector>
__global__ void __launch_bounds__(RAY_MAX_THREADS)
k_ray_update(MapGeom geom, ScanDevice scan, const ParticleResult* __restrict__ results, uint32_t first_particle,
             const uint32_t* __restrict__ alive_list,
             const int32_t* __restrict__ slot_of, uint32_t* __restrict__ cells, SlotMeta* __restrict__ meta,
             uint32_t* __restrict__ bands_all, size_t cells_per_grid, int radius, int reach, StepCounters* counters) {
    extern __shared__ __align__(16) uint32_t s_win[];
    __shared__ int s_blo[RAY_MAX_BANDS], s_bhi[RAY_MAX_BANDS];
    __shared__ int s_row_off[RAY_MAX_ROWS + 1];   // first window cell of each row (+ total at [wh])
    __shared__ int s_row_x[RAY_MAX_ROWS];         // x0 | (width << 16)
    __shared__ int s_ext[4];
    if ((unsigned long long)blockIdx.x >= counters->n_alive) return;
    const uint32_t p = alive_list[blockIdx.x];
    ext_init(s_ext);
    const ParticleResult r = results[first_particle + p];
    const float px = r.x, py = r.y, ptheta = r.theta;
    uint32_t* grid = cells + (size_t)slot_of[p] * cells_per_grid;

    // Map::integrate, map.rs:71-73: ray start in grid coordinates
    const float sx = world_to_grid(px, geom.pos_x, geom.res);
    const float sy = world_to_grid(py, geom.pos_y, geom.res);
    const long long lcx = f32_as_isize(floorf(sx)), lcy = f32_as_isize(floorf(sy));
    // every ray starts in the same cell; outside the grid nothing is emitted (ray.rs:88-92)
    if (lcx < 0 || lcx >= (long long)geom.gw || lcy < 0 || lcy >= (long long)geom.gh) return;
    const int cx = (int)lcx, cy = (int)lcy;
    if (window_would_overflow(geom, &meta[slot_of[p]], cx, cy, reach)) {
        if (threadIdx.x == 0) atomicAdd(&counters->window_overflow, 1ull);
        return;   // the grid is left as it was; the step reports SLAMRS_E_WINDOW
    }
    uint32_t* bands = bands_all + (size_t)slot_of[p] * bands_per_slot(geom);
    band_init(s_blo, s_bhi);

    // ---- row table of the disc window, clipped to the grid
    const int wy0 = max(0, cy - radius), wy1 = min((int)geom.gh, cy + radius + 1);
    const int band0 = wy0 / BAND_ROWS;
    const int wh = wy1 - wy0;
    for (int ly = threadIdx.x; ly < wh; ly += blockDim.x) {
        const int dy = wy0 + ly - cy;
        const int hw = isqrt_small(radius * radius - dy * dy);
        int x0 = max(0, cx - hw), x1 = min((int)geom.gw, cx + hw + 1);
        if (kVector) {
            x0 &= ~3;
            x1 = min((int)geom.gw, (x1 + 3) & ~3);
        }
        s_row_x[ly] = x0 | ((x1 - x0) << 16);
    }
    __syncthreads();
    if (threadIdx.x < 32) {  // exclusive prefix sum of the row widths, 32 rows per round
        int carry = 0;
        for (int base = 0; base < wh; base += 32) {
            const int ly = base + (int)threadIdx.x;
            const int w = ly < wh ? (s_row_x[ly] >> 16) : 0;
            int inc = w;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int t = __shfl_up_sync(0xffffffffu, inc, o);
                if ((int)threadIdx.x >= o) inc += t;
            }
            if (ly < wh) s_row_off[ly] = carry + inc - w;
            carry += __shfl_sync(0xffffffffu, inc, 31);
        }
        if (threadIdx.x == 0) s_row_off[wh] = carry;
    }
    __syncthreads();
    const int wcells = s_row_off[wh];

    if (kVector) {
        uint4* w4 = reinterpret_cast<uint4*>(s_win);
        for (int i = threadIdx.x; i < (wcells >> 2); i += blockDim.x) w4[i] = make_uint4(0u, 0u, 0u, 0u);
    } else {
        for (int i = threadIdx.x; i < wcells; i += blockDim.x) s_win[i] = 0u;
    }
    __syncthreads();

    bool saturated = false;
    uint32_t spilled = 0;
    ZeroLengthHits zero_length;
    for (uint32_t t = threadIdx.x; t < scan.n_beams; t += blockDim.x) {
        const uint32_t b = scan.order ? scan.order[t] : t;
        const float dist = scan.dist[b];
        float ex, ey;
        beam_endpoint(px, py, ptheta, scan.angle[b], dist, &ex, &ey);
        const float gx = world_to_grid(ex, geom.pos_x, geom.res);
        const float gy = world_to_grid(ey, geom.pos_y, geom.res);
        // measured distance in cells (map.rs:84) and the per-ray form of inverse_sensor_model
        const RayClassifier cls = make_ray_classifier(__fdiv_rn(dist, geom.res), scan.valid[b] != 0);
        if (fabsf(__fsub_rn(gx, sx)) == 0.0f && fabsf(__fsub_rn(gy, sy)) == 0.0f) {
            // zero-length ray (see ZeroLengthHits): its hits would overflow a 16-bit half of the window
            const float dxs = __fsub_rn(sx, __fadd_rn((float)cx, 0.5f)), dys = __fsub_rn(sy, __fadd_rn((float)cy, 0.5f));
            zero_length.tally(cls, __fadd_rn(__fmul_rn(dxs, dxs), __fmul_rn(dys, dys)));
            continue;
        }
        // apply_measurement, map.rs:88-106 (additional_steps = 2)
        ray_walk_acc(sx, sy, gx, gy, geom.gw, geom.gh, 2u, [&](int x, int y, float acc) {
            const uint32_t inc = classify_cell(cls, acc);
            if (inc != 0u) {
                const int ly = y - wy0;
                bool in_window = false;
                if ((unsigned)ly < (unsigned)wh) {
                    const int rx = s_row_x[ly];
                    const int lx = x - (rx & 0xffff);
                    if ((unsigned)lx < (unsigned)(rx >> 16)) {
                        atomicAdd(&s_win[s_row_off[ly] + lx], inc);
                        in_window = true;
                    }
                }
                if (!in_window) {  // beyond the window (range larger than shared memory allows)
                    global_cell_add(&grid[phys_index(geom, (uint32_t)x, (uint32_t)y)], inc, &saturated);
                    ext_add(s_ext, x, y, x, y);
                    band_add(s_blo, s_bhi, band0, y, x, x);
                    band_add_global(bands, geom, band0, x, y);
                    spilled++;
                }
            }
        });
    }
    {
        auto exact_add = [&](int x, int y, uint32_t inc) {
            global_cell_add(&grid[phys_index(geom, (uint32_t)x, (uint32_t)y)], inc, &saturated);
        };
        spilled += zero_length.flush(cx, cy, exact_add, s_ext, s_blo, s_bhi, band0);
    }
    __syncthreads();

    // ---- write-back: grid += window, saturating per 16-bit counter, untouched groups skipped.
    // RAY_WB_BATCH independent global loads are issued per thread before the first dependent store.
    int exmin = 0x7fffffff, eymin = 0x7fffffff, exmax = -1, eymax = -1;   // this thread's touched extent
    if (kVector) {
        const int total4 = wcells >> 2;
        const uint4* win4 = reinterpret_cast<const uint4*>(s_win);
        for (int base = threadIdx.x; base < total4; base += blockDim.x * RAY_WB_BATCH) {
            uint4 d[RAY_WB_BATCH], v[RAY_WB_BATCH];
            uint4* gp[RAY_WB_BATCH];
            bool nz[RAY_WB_BATCH];
#pragma unroll
            for (int j = 0; j < RAY_WB_BATCH; ++j) {
                const int i = base + j * (int)blockDim.x;
                nz[j] = false;
                if (i < total4) {
                    d[j] = win4[i];
                    nz[j] = (d[j].x | d[j].y | d[j].z | d[j].w) != 0u;
                    if (nz[j]) {
                        int lo = 0, hi = wh;   // row containing window cell 4*i
                        while (hi - lo > 1) {
                            const int mid = (lo + hi) >> 1;
                            if (s_row_off[mid] <= 4 * i) lo = mid; else hi = mid;
                        }
                        const int lx = 4 * i - s_row_off[lo];
                        const int gx0 = (s_row_x[lo] & 0xffff) + lx;
                        exmin = min(exmin, gx0); exmax = max(exmax, gx0 + 3);
                        eymin = min(eymin, wy0 + lo); eymax = max(eymax, wy0 + lo);
                        band_add(s_blo, s_bhi, band0, wy0 + lo, gx0, gx0 + 3);
                        gp[j] = reinterpret_cast<uint4*>(grid + phys_index(geom, (uint32_t)gx0, (uint32_t)(wy0 + lo)));
                    }
                }
            }
#pragma unroll
            for (int j = 0; j < RAY_WB_BATCH; ++j)
                if (nz[j]) v[j] = *gp[j];
#pragma unroll
            for (int j = 0; j < RAY_WB_BATCH; ++j) {
                if (nz[j]) {
                    v[j].x = cell_sat_add(v[j].x, d[j].x, &saturated);
                    v[j].y = cell_sat_add(v[j].y, d[j].y, &saturated);
                    v[j].z = cell_sat_add(v[j].z, d[j].z, &saturated);
                    v[j].w = cell_sat_add(v[j].w, d[j].w, &saturated);
                    *gp[j] = v[j];
                }
            }
        }
    } else {
        for (int ly = threadIdx.x >> 5; ly < wh; ly += blockDim.x >> 5) {
            const int rx = s_row_x[ly], x0 = rx & 0xffff, w = rx >> 16, off = s_row_off[ly];
            for (int c = threadIdx.x & 31; c < w; c += 32) {
                const uint32_t d = s_win[off + c];
                if (d != 0u) {
                    uint32_t* g = grid + phys_index(geom, (uint32_t)(x0 + c), (uint32_t)(wy0 + ly));
                    *g = cell_sat_add(*g, d, &saturated);
                    exmin = min(exmin, x0 + c); exmax = max(exmax, x0 + c);
                    eymin = min(eymin, wy0 + ly); eymax = max(eymax, wy0 + ly);
                    band_add(s_blo, s_bhi, band0, wy0 + ly, x0 + c, x0 + c);
                }
            }
        }
    }
    ext_add(s_ext, exmin, eymin, exmax, eymax);
    __syncthreads();
    band_commit(s_blo, s_bhi, band0, bands, geom);
    if (threadIdx.x == 0) ext_commit(s_ext, &meta[slot_of[p]], (int)geom.gw);
    if (saturated) atomicAdd(&counters->saturated, 1ull);
    if (spilled) atomicAdd(&counters->spilled, (unsigned long long)spilled);
}

// one 8-cell group as a single 256-bit access (coherent: the exact path may have written the cell)
__device__ __forceinline__ void ld_group_v8(const uint4* p, uint4& a, uint4& b) {
    asm volatile("ld.global.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(a.x), "=r"(a.y), "=r"(a.z), "=r"(a.w), "=r"(b.x), "=r"(b.y), "=r"(b.z), "=r"(b.w)
                 : "l"(p) : "memory");
}
__device__ __forceinline__ void st_group_v8(uint4* p, const uint4& a, const uint4& b) {
    asm volatile("st.global.v8.u32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "r"(a.x), "r"(a.y), "r"(a.z), "r"(a.w),
                 "r"(b.x), "r"(b.y), "r"(b.z), "r"(b.w) : "memory");
}

// ------------------------------------------------------------------------------- packed variant
// Same algorithm with a 2-byte window cell: bits 0..10 = free hits (a cell can be crossed by at
// most n_beams <= 2047 rays per scan), bits 11..15 = occupied hits (<= 31; a 32nd hit in one scan
// takes the exact global path). Half the shared memory per particle => two CTAs per SM at a 6 m /
// 5 cm window, which is what hides the latency of the serial cell walk. Free hits (the vast
// majority) are single fire-and-forget shared-memory adds; the walk itself is written with the
// row lookup hoisted to y-steps.
constexpr uint32_t PK_FREE_BITS = 11;
constexpr uint32_t PK_FREE_MASK = (1u << PK_FREE_BITS) - 1u;
constexpr uint32_t PK_OCC_MAX = 31;
constexpr uint32_t RAY_PACKED_MAX_BEAMS = PK_FREE_MASK;

__host__ __device__ inline int ray_window_cells_upper_bound_packed(int radius) {
    int total = 0;
    for (int dy = -radius; dy <= radius; ++dy) total += 2 * isqrt_small(radius * radius - dy * dy) + 1 + 14;
    return total;
}

// Facts the packed kernels' fast walk relies on (see DESIGN.md):
//  * |x0 - centre_x| and |y0 - centre_y| never decrease along a walk (x only moves by x_inc, y
//    only by y_inc, away from the start cell), IEEE rounding is monotone, so
//    acc = fl(fl(dx^2) + fl(dy^2)) is non-decreasing along the ray. The inverse sensor model is
//    therefore a free run (acc < free_below), then an occupied run (acc <= prior_above, hits
//    only), then prior cells that add nothing: two tight loops and an early exit replace the
//    per-cell three-way classification.
//  * a ray whose endpoint cell is (ax, ay) cells away from the start cell visits only cells within
//    (ax + 2, ay + 2) of it; if that corner is inside the disc window and the disc is inside the
//    grid, no per-cell window or grid test is needed.
//
// At most RAY_OCC_PER_RAY_MAX = 7 cells of one ray are occupied. In cell units, let S be the start point, u the
// unit direction of the ray, d the measured distance, E the endpoint (|E - S| = d). The iterator visits the cells the
// line S + t u passes through, in order of t, one grid line per step: up to the endpoint cell the cells it meets for
// t in [0, d], then additional_steps = 2 more. A cell is occupied when its centre c has |c - S| in [d - 1, d + 1]
// (map.rs:148-172, tolerance 2). Every point p of the cell is within sqrt(2)/2 of c, so the line meets an occupied
// cell at some t = |p - S| >= d - 1 - sqrt(2)/2. The occupied cells up to the endpoint cell therefore all meet the
// line in [d - 1.71, d]: one cell plus one per grid line crossed inside that interval, which holds fewer than
// 1.71 |u_x| + 1 vertical and 1.71 |u_y| + 1 horizontal lines, at most 1.71 sqrt(2) + 2 = 4.42 together: at most
// 4 crossings, 5 cells. With the 2 cells after the endpoint cell: 7. A zero-length ray parks 3 hits. The walk's f32
// rounding moves a step by far less than a cell at these distances; tests/test_ray_bypass_bounds.py searches a lattice
// of start offsets, headings and distances with the reference's walk and finds at most 5.
//
// So one work item parks at most 7 hits per ray of its half: RAY_SPILL_CAP entries. The lower half's parked hits on
// the start row, all of them occupied hits of window cells, travel to the upper half as 16-bit counts per start-row
// cell (HalfXchg::occ): at most 7 x 2,047 < 65,536 of them.
constexpr uint32_t RAY_OCC_PER_RAY_MAX = 7;
constexpr uint32_t RAY_SPILL_CAP = RAY_OCC_PER_RAY_MAX * RAY_PACKED_MAX_BEAMS;
static_assert(RAY_SPILL_CAP <= 0xffffu, "a start-row count of parked hits is 16 bits");
// SLAMRS_RAY_TRACE (tuning builds): thread 0 of every CTA adds the cycles it spent per phase of an item
#ifdef SLAMRS_RAY_TRACE
__device__ unsigned long long g_ray_trace[16];
#define RAY_STAMP(k) do { if (threadIdx.x == 0) { const long long _t = clock64(); atomicAdd(&g_ray_trace[k], (unsigned long long)(_t - t_prev)); t_prev = _t; } } while (0)
#else
#define RAY_STAMP(k) do { } while (0)
#endif
#ifdef SLAMRS_RAY_TRACE
__device__ unsigned long long g_ray_trace_items[2];
// per work item of the LAST launch: globaltimer (ns) at each phase boundary of k_ray_update_half, + SM id and kind
constexpr int RAY_LOG_ITEMS = 16384, RAY_LOG_COLS = 16;
__device__ unsigned long long g_ray_log[RAY_LOG_ITEMS * RAY_LOG_COLS];
__device__ __forceinline__ unsigned long long ray_gtime() { unsigned long long t; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t)); return t; }
__device__ __forceinline__ unsigned ray_smid() { unsigned r; asm volatile("mov.u32 %0, %smid;" : "=r"(r)); return r; }
#define RAY_LOG(w, k) do { if (threadIdx.x == 0 && (w) < (unsigned long long)RAY_LOG_ITEMS) g_ray_log[(w) * RAY_LOG_COLS + (k)] = ray_gtime(); } while (0)
#define RAY_LOG_V(w, k, v) do { if (threadIdx.x == 0 && (w) < (unsigned long long)RAY_LOG_ITEMS) g_ray_log[(w) * RAY_LOG_COLS + (k)] = (v); } while (0)
#else
#define RAY_LOG(w, k) do { } while (0)
#define RAY_LOG_V(w, k, v) do { } while (0)
#endif

// The walk of one particle's beams into the 16-bit shared-memory window (GridRayIterator, ray.rs:21-110, with the
// inverse sensor model of map.rs:148-172), shared by k_ray_update_packed (every beam, `beams` = scan.order or null
// for identity order) and k_ray_update_half (this half's list). `disc_in_grid`: the window holds every in-grid cell
// within `rad` of the start cell in the rows this walk can reach. Out of line on purpose: compiled on its own the
// free-run loop stays the 25-instruction predicated block tools/sass_hot_loop.py checks for.
//
// Hits that bypass the window (the 32nd occupied hit of a cell in one scan, zero-length rays, and cells outside
// the window) take the exact path. kParkBypass: they are parked in my_spill and applied after the write-back --
// a clone's own slot receives its cells only then; at most RAY_OCC_PER_RAY_MAX occupied cells per ray (3 hits of a
// zero-length ray), so RAY_SPILL_CAP entries suffice when the window holds every cell a ray reaches.
// Otherwise they go straight to the grid with a saturating CAS, widening the slot's band table where the window's
// bands do not cover them.
template <bool kParkBypass>
__device__ __noinline__ void ray_walk_packed(const MapGeom& geom, const ScanDevice& scan, const uint16_t* beams, uint32_t n_walk,
                                             float px, float py, float ptheta, float sx, float sy, int cx0, int cy0, int rad,
                                             bool disc_in_grid, int wy0, int wh, int band0, uint32_t* s_win, const int2* s_row,
                                             const uint32_t* s_rowb, int* s_blo, int* s_bhi, int* s_ext,
                                             uint32_t* __restrict__ grid, uint32_t* __restrict__ bands, uint32_t* s_nspill_p,
                                             uint32_t* __restrict__ my_spill, bool* saturated_p, uint32_t* spilled_p,
                                             uint32_t* cell_steps_p) {
    const int gw = (int)geom.gw, gh = (int)geom.gh;
    const uint32_t win_base = (uint32_t)__cvta_generic_to_shared(s_win);
    bool saturated = false;
    uint32_t spilled = 0, cell_steps = 0;
    ZeroLengthHits zero_length;
    auto exact_add = [&](int x, int y, uint32_t inc) {
        if constexpr (kParkBypass) {
            const uint32_t k = atomicAdd(s_nspill_p, 1u);
            if (k < RAY_SPILL_CAP) my_spill[k] = (uint32_t)x | ((uint32_t)y << 15) | (inc == CELL_OCC_INC ? 0x40000000u : 0u);
        } else {
            global_cell_add(&grid[phys_index(geom, (uint32_t)x, (uint32_t)y)], inc, &saturated);
        }
    };
    // The row table is read at every y-step of the walk. Its shared address is kept in a register the
    // compiler cannot re-derive: left to itself ptxas may rebuild it inside the loop (S2UR + ULEA per
    // step, seen in SASS after an unrelated change elsewhere in the kernel), which costs the walk ~15 %.
    uint32_t rowb_base = (uint32_t)__cvta_generic_to_shared(s_rowb);
    asm volatile("" : "+r"(rowb_base));
    auto load_rowb = [&](int row) {
        uint32_t v;
        asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(rowb_base + 4u * (uint32_t)row) : "memory");
        return v;
    };
    for (uint32_t t = threadIdx.x; t < n_walk; t += blockDim.x) {
        const uint32_t b = beams ? beams[t] : t;
        const float dist = scan.dist[b];
        float ex, ey;
        beam_endpoint(px, py, ptheta, scan.angle[b], dist, &ex, &ey);
        const float x1 = world_to_grid(ex, geom.pos_x, geom.res);
        const float y1 = world_to_grid(ey, geom.pos_y, geom.res);
        const RayClassifier cls = make_ray_classifier(__fdiv_rn(dist, geom.res), scan.valid[b] != 0);

        // GridRayIterator::new (ray.rs:21-77) -- identical arithmetic to ray_walk_acc
        const float delta_x = fabsf(__fsub_rn(x1, sx)), delta_y = fabsf(__fsub_rn(y1, sy));
        const float fx0 = floorf(sx), fy0 = floorf(sy);
        unsigned long long n = 1ull + 2ull;   // additional_steps = 2 (map.rs:97)
        unsigned long long ax = 0ull, ay = 0ull;   // |endpoint cell - start cell| per axis
        int x_inc, y_inc;
        float error;
        if (delta_x == 0.0f) {
            x_inc = 0;
            error = __int_as_float(0x7f800000);
        } else if (x1 > sx) {
            x_inc = 1;
            ax = (unsigned long long)f32_as_isize(__fsub_rn(floorf(x1), (float)cx0));
            error = __fmul_rn(__fsub_rn(__fadd_rn(fx0, 1.0f), sx), delta_y);
        } else {
            x_inc = -1;
            ax = (unsigned long long)(long long)cx0 - (unsigned long long)f32_as_isize(floorf(x1));
            error = __fmul_rn(__fsub_rn(sx, fx0), delta_y);
        }
        if (delta_y == 0.0f) {
            y_inc = 0;
            error = __fsub_rn(error, __int_as_float(0x7f800000));
        } else if (y1 > sy) {
            y_inc = 1;
            ay = (unsigned long long)f32_as_isize(floorf(y1)) - (unsigned long long)(long long)cy0;
            error = __fsub_rn(error, __fmul_rn(__fsub_rn(__fadd_rn(fy0, 1.0f), sy), delta_x));
        } else {
            y_inc = -1;
            ay = (unsigned long long)(long long)cy0 - (unsigned long long)f32_as_isize(floorf(y1));
            error = __fsub_rn(error, __fmul_rn(__fsub_rn(sy, fy0), delta_x));
        }
        n += ax + ay;   // wrapping isize arithmetic, then `as usize`
        const unsigned long long cap = (unsigned long long)geom.gw + geom.gh + 8ull;
        int remaining = (int)(n < cap ? n : cap);
        cell_steps += (uint32_t)remaining;   // what the reference's iterator would visit; minus the rest if the ray leaves the grid

        const float x_step = (float)x_inc, y_step = (float)y_inc;
        float cxf = __fadd_rn((float)cx0, 0.5f), cyf = __fadd_rn((float)cy0, 0.5f);
        float dxs = __fsub_rn(sx, cxf), dys = __fsub_rn(sy, cyf);
        float dx2 = __fmul_rn(dxs, dxs), dy2 = __fmul_rn(dys, dys);
        if (delta_x == 0.0f && delta_y == 0.0f) {   // see ZeroLengthHits
            zero_length.tally(cls, __fadd_rn(dx2, dy2));
            continue;
        }

        // every cell of this ray inside the window and the grid?
        bool fast = false;
        if (disc_in_grid && ax < 4096ull && ay < 4096ull) {
            const int cxa = (int)ax + 2, cya = (int)ay + 2;
            fast = cxa * cxa + cya * cya <= rad * rad;
        }
        if (fast) {
            uint32_t x2 = 2u * (uint32_t)cx0;         // twice the current column
            const uint32_t x_inc2 = (uint32_t)(2 * x_inc);
            int ly = cy0 - wy0;
            uint32_t rb = load_rowb(ly);
            // The first cells of a walk are free whatever its direction: the cell reached after k steps is k cells from
            // the start cell in the Manhattan sense, the start point lies inside the start cell, so both offsets to the
            // cell centre are at most (cells + 0.5) and acc <= (k + 0.5)^2 + 0.25 < K^2 for k < K; with K^2 <= 0.999 x
            // free_below (the margin dwarfs the f32 rounding of acc) those K cells pass `acc < free_below` without
            // evaluating it. They take a loop without the distance arithmetic; the distance state is then rebuilt from
            // the cell position -- cxf and cyf only ever held (integer + 0.5) exactly, so the rebuilt values are the
            // accumulated ones bit for bit -- and the free run continues with the test.
            {
                const float kf = floorf(__fsqrt_rn(__fmul_rn(cls.free_below, 0.999f)));
                int safe = (kf >= 1.0f && kf < 1.0e6f) ? (int)kf : 0;      // (NaN and tiny thresholds: none)
                safe = min(safe, remaining);
                remaining -= safe;
                for (; safe > 0; --safe) {
                    const uint32_t c2 = rb + x2;
                    asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(c2 & ~3u), "r"((c2 & 2u) ? 0x10000u : 1u) : "memory");
                    if (error > 0.0f) {
                        error = __fsub_rn(error, delta_x);
                        ly += y_inc;
                        rb = load_rowb(ly);
                    } else {
                        error = __fadd_rn(error, delta_y);
                        x2 += x_inc2;
                    }
                }
                cxf = __fadd_rn((float)(x2 >> 1), 0.5f);
                cyf = __fadd_rn((float)(wy0 + ly), 0.5f);
                dxs = __fsub_rn(sx, cxf); dys = __fsub_rn(sy, cyf);
                dx2 = __fmul_rn(dxs, dxs); dy2 = __fmul_rn(dys, dys);
            }
            while (remaining > 0) {                    // free run
                const float acc = __fadd_rn(dx2, dy2);
                if (!(acc < cls.free_below)) break;
                const uint32_t c2 = rb + x2;           // shared byte address of the 16-bit window cell
                asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(c2 & ~3u), "r"((c2 & 2u) ? 0x10000u : 1u) : "memory");
                if (error > 0.0f) {
                    error = __fsub_rn(error, delta_x);
                    cyf = __fadd_rn(cyf, y_step);
                    dys = __fsub_rn(sy, cyf);
                    dy2 = __fmul_rn(dys, dys);
                    ly += y_inc;
                    rb = load_rowb(ly);
                } else {
                    error = __fadd_rn(error, delta_y);
                    cxf = __fadd_rn(cxf, x_step);
                    dxs = __fsub_rn(sx, cxf);
                    dx2 = __fmul_rn(dxs, dxs);
                    x2 += x_inc2;
                }
                remaining -= 1;
            }
            if (cls.mid_inc != 0u) {                   // occupied run (hits only): bounded 5-bit field, exact path beyond it
                while (remaining > 0) {
                    const float acc = __fadd_rn(dx2, dy2);
                    if (acc > cls.prior_above) break;
                    const uint32_t c2 = rb + x2;
                    const uint32_t shift = ((c2 & 2u) << 3) + PK_FREE_BITS;
                    uint32_t old;
                    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(old) : "r"(c2 & ~3u) : "memory");
                    bool done_here = false;
                    for (;;) {
                        if (((old >> shift) & PK_OCC_MAX) == PK_OCC_MAX) break;
                        uint32_t seen;
                        asm volatile("atom.shared.cas.b32 %0, [%1], %2, %3;"
                                     : "=r"(seen) : "r"(c2 & ~3u), "r"(old), "r"(old + (1u << shift)) : "memory");
                        if (seen == old) { done_here = true; break; }
                        old = seen;
                    }
                    if (!done_here) {
                        const int x = (int)(x2 >> 1), y = wy0 + ly;
                        exact_add(x, y, CELL_OCC_INC);
                        ext_add(s_ext, x, y, x, y);
                        band_add(s_blo, s_bhi, band0, y, x, x);
                        spilled++;
                    }
                    if (error > 0.0f) {
                        error = __fsub_rn(error, delta_x);
                        cyf = __fadd_rn(cyf, y_step);
                        dys = __fsub_rn(sy, cyf);
                        dy2 = __fmul_rn(dys, dys);
                        ly += y_inc;
                        rb = load_rowb(ly);
                    } else {
                        error = __fadd_rn(error, delta_y);
                        cxf = __fadd_rn(cxf, x_step);
                        dxs = __fsub_rn(sx, cxf);
                        dx2 = __fmul_rn(dxs, dxs);
                        x2 += x_inc2;
                    }
                    remaining -= 1;
                }
            }
            continue;
        }

        // general walk: per-cell window and grid tests (rays that may leave the window or the grid)
        int x = cx0, y = cy0;
        int ly = y - wy0;
        int2 row = s_row[ly];                      // the start cell is always inside the window
        int lx = x - (row.y & 0xffff);
        int row_w = row.y >> 16;
        bool inside = true;
        while (remaining > 0 && inside) {
            const float acc = __fadd_rn(dx2, dy2);
            const bool is_free = acc < cls.free_below;
            const bool is_mid = !is_free && !(acc > cls.prior_above) && (cls.mid_inc != 0u);
            if (is_free | is_mid) {
                const bool in_win = (unsigned)lx < (unsigned)row_w;
                const int cell = row.x + lx;
                const uint32_t addr = win_base + ((uint32_t)(cell >> 1) << 2);
                const uint32_t shift = (cell & 1) << 4;
                if (is_free & in_win) {
                    asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(addr), "r"(1u << shift) : "memory");
                } else {
                    bool done_here = false;
                    if (in_win) {   // occupied hit: bounded 5-bit field, exact path when it would overflow
                        uint32_t* wp = &s_win[cell >> 1];
                        uint32_t old = *wp;
                        for (;;) {
                            if (((old >> (shift + PK_FREE_BITS)) & PK_OCC_MAX) == PK_OCC_MAX) break;
                            const uint32_t seen = atomicCAS(wp, old, old + (1u << (shift + PK_FREE_BITS)));
                            if (seen == old) { done_here = true; break; }
                            old = seen;
                        }
                    }
                    if (!done_here) {
                        exact_add(x, y, is_free ? CELL_FREE_INC : CELL_OCC_INC);
                        ext_add(s_ext, x, y, x, y);
                        band_add(s_blo, s_bhi, band0, y, x, x);
                        if constexpr (!kParkBypass) band_add_global(bands, geom, band0, x, y);
                        spilled++;
                    }
                }
            }
            if (error > 0.0f) {                    // GridRayIterator::next (ray.rs:96-104)
                y += y_inc;
                error = __fsub_rn(error, delta_x);
                cyf = __fadd_rn(cyf, y_step);
                dys = __fsub_rn(sy, cyf);
                dy2 = __fmul_rn(dys, dys);
                inside = (unsigned)y < (unsigned)gh;
                ly += y_inc;
                if ((unsigned)ly < (unsigned)wh) {
                    row = s_row[ly];
                    row_w = row.y >> 16;
                    lx = x - (row.y & 0xffff);
                } else {
                    row_w = 0;
                }
            } else {
                x += x_inc;
                error = __fadd_rn(error, delta_y);
                cxf = __fadd_rn(cxf, x_step);
                dxs = __fsub_rn(sx, cxf);
                dx2 = __fmul_rn(dxs, dxs);
                inside = (unsigned)x < (unsigned)gw;
                lx += x_inc;
            }
            remaining -= 1;
        }
        cell_steps -= (uint32_t)remaining;   // the walk ended at the grid border
    }
    spilled += zero_length.flush(cx0, cy0, exact_add, s_ext, s_blo, s_bhi, band0);
    if (saturated) *saturated_p = true;
    *spilled_p += spilled;
    *cell_steps_p += cell_steps;
}

// Adds one 8-cell group of the packed window (d: eight 16-bit cells) to the grid's eight counters (va, vb). The
// window value is unpacked without a branch; only a grid counter at or above 2^15 (which one scan's increment could
// saturate) takes the saturating form.
__device__ __forceinline__ uint32_t unpack_window_cell(uint32_t packed16) {
    return (packed16 & PK_FREE_MASK) | ((packed16 >> PK_FREE_BITS) << 16);
}
__device__ __forceinline__ void merge_window_group(uint4& va, uint4& vb, const uint4& d, bool* saturated) {
    const uint32_t high_any = (va.x | va.y | va.z | va.w | vb.x | vb.y | vb.z | vb.w) & 0x80008000u;
    if (high_any == 0u) {
        va.x += unpack_window_cell(d.x & 0xffffu); va.y += unpack_window_cell(d.x >> 16);
        va.z += unpack_window_cell(d.y & 0xffffu); va.w += unpack_window_cell(d.y >> 16);
        vb.x += unpack_window_cell(d.z & 0xffffu); vb.y += unpack_window_cell(d.z >> 16);
        vb.z += unpack_window_cell(d.w & 0xffffu); vb.w += unpack_window_cell(d.w >> 16);
    } else {
        va.x = cell_sat_add(va.x, unpack_window_cell(d.x & 0xffffu), saturated); va.y = cell_sat_add(va.y, unpack_window_cell(d.x >> 16), saturated);
        va.z = cell_sat_add(va.z, unpack_window_cell(d.y & 0xffffu), saturated); va.w = cell_sat_add(va.w, unpack_window_cell(d.y >> 16), saturated);
        vb.x = cell_sat_add(vb.x, unpack_window_cell(d.z & 0xffffu), saturated); vb.y = cell_sat_add(vb.y, unpack_window_cell(d.z >> 16), saturated);
        vb.z = cell_sat_add(vb.z, unpack_window_cell(d.w & 0xffffu), saturated); vb.w = cell_sat_add(vb.w, unpack_window_cell(d.w >> 16), saturated);
    }
}

// Work distribution of both packed kernels. A kernel is launched with as many CTAs as are resident at once and
// every CTA pops work items from an atomic counter until the list is empty: the list holds the few hundred
// particles that survive this step's resampling, not the whole population.
//
// k_ray_update_packed: a whole particle per work item (two CTAs per SM at a 6 m / 5 cm window), for row-major and
// windowed slots. Its items come from the survivor list alone; the particle's slot is its own, so the window is
// written back into it in place.
__global__ void __maxnreg__(80)   // 2 CTAs of 384 threads per SM; blocks have at most RAY_MAX_THREADS threads
k_ray_update_packed(MapGeom geom, ScanDevice scan, const ParticleResult* __restrict__ results, uint32_t first_particle,
                    const uint32_t* __restrict__ alive_list, const int32_t* __restrict__ slot_of, uint32_t* __restrict__ cells,
                    SlotMeta* __restrict__ meta, uint32_t* __restrict__ bands_all, size_t cells_per_grid, int radius, int reach,
                    StepCounters* counters) {
    extern __shared__ __align__(16) uint32_t s_win[];   // two 16-bit cells per word
    __shared__ int s_blo[RAY_MAX_BANDS], s_bhi[RAY_MAX_BANDS];
    __shared__ int2 s_row[RAY_MAX_ROWS + 1];            // .x = first window cell of the row, .y = x0 | width << 16
    __shared__ uint32_t s_rowb[RAY_MAX_ROWS];           // shared byte address of column x = 0 of the row
    __shared__ int s_ext[4];
    __shared__ unsigned long long s_next;
    const unsigned long long n_items = counters->n_alive;
    const int gw = (int)geom.gw, gh = (int)geom.gh;
    const uint32_t win_base = (uint32_t)__cvta_generic_to_shared(s_win);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, n_warps = blockDim.x >> 5;
    const uint32_t n_bands_slot = bands_per_slot(geom);
    bool saturated = false;
    uint32_t spilled = 0;
    uint32_t cell_steps = 0;   // iterator steps of this thread's rays (SURVEY.md 8(d): C_p, the unit of the ray update's bytes)

#ifdef SLAMRS_RAY_TRACE
    long long t_prev = clock64();
#endif
    for (;;) {
        __syncthreads();       // the previous item's shared state is no longer read
        RAY_STAMP(0);
        if (threadIdx.x == 0) s_next = atomicAdd(&counters->ray_work_head, 1ull);
        __syncthreads();
        const unsigned long long item = s_next;
        if (item >= n_items) break;
        const uint32_t p = alive_list[item];
        const int32_t slot = slot_of[p];
        uint32_t* grid = cells + (size_t)slot * cells_per_grid;
        ext_init(s_ext);
        const ParticleResult r = results[first_particle + p];
        const float px = r.x, py = r.y, ptheta = r.theta;

        const float sx = world_to_grid(px, geom.pos_x, geom.res);
        const float sy = world_to_grid(py, geom.pos_y, geom.res);
        const long long lcx = f32_as_isize(floorf(sx)), lcy = f32_as_isize(floorf(sy));
        // every ray starts in the same cell; outside the grid nothing is emitted (ray.rs:88-92)
        const bool start_inside = !(lcx < 0 || lcx >= (long long)geom.gw || lcy < 0 || lcy >= (long long)geom.gh);
        if (!start_inside) continue;
        const int cx0 = (int)lcx, cy0 = (int)lcy;
        if (window_would_overflow(geom, &meta[slot], cx0, cy0, reach)) {   // windowed slots only
            if (threadIdx.x == 0) atomicAdd(&counters->window_overflow, 1ull);
            continue;   // the grid is left as it was; the step reports SLAMRS_E_WINDOW
        }
        uint32_t* bands = bands_all + (size_t)slot * n_bands_slot;
        band_init(s_blo, s_bhi);

        // ---- row table of the disc window (x ranges aligned to 8 cells = one 128-bit group)
        const int wy0 = max(0, cy0 - radius), wy1 = min(gh, cy0 + radius + 1);
        const int band0 = wy0 / BAND_ROWS;
        const int wh = wy1 - wy0;
        for (int ly = threadIdx.x; ly < wh; ly += blockDim.x) {
            const int dy = wy0 + ly - cy0;
            const int hw = isqrt_small(radius * radius - dy * dy);
            const int x0 = max(0, cx0 - hw) & ~7;
            const int x1 = min(gw, (min(gw, cx0 + hw + 1) + 7) & ~7);
            s_row[ly].y = x0 | ((x1 - x0) << 16);
        }
        __syncthreads();
        if (threadIdx.x < 32) {
            int carry = 0;
            for (int base = 0; base < wh; base += 32) {
                const int ly = base + (int)threadIdx.x;
                const int w = ly < wh ? (s_row[ly].y >> 16) : 0;
                int inc = w;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const int t = __shfl_up_sync(0xffffffffu, inc, o);
                    if ((int)threadIdx.x >= o) inc += t;
                }
                if (ly < wh) {
                    const int first = carry + inc - w;
                    s_row[ly].x = first;
                    s_rowb[ly] = win_base + 2u * (uint32_t)(first - (s_row[ly].y & 0xffff));
                }
                carry += __shfl_sync(0xffffffffu, inc, 31);
            }
            if (threadIdx.x == 0) s_row[wh] = make_int2(carry, 0);
        }
        __syncthreads();
        const int wcells = s_row[wh].x;
        {
            uint4* w4 = reinterpret_cast<uint4*>(s_win);
            for (int i = threadIdx.x; i < (wcells >> 3); i += blockDim.x) w4[i] = make_uint4(0u, 0u, 0u, 0u);
        }
        __syncthreads();

        RAY_STAMP(1);
        const bool disc_in_grid = cx0 - radius >= 0 && cx0 + radius < gw && cy0 - radius >= 0 && cy0 + radius < gh;
        ray_walk_packed<false>(geom, scan, scan.order, scan.n_beams, px, py, ptheta, sx, sy, cx0, cy0, radius, disc_in_grid, wy0,
                               wh, band0, s_win, s_row, s_rowb, s_blo, s_bhi, s_ext, grid, bands, nullptr, nullptr, &saturated,
                               &spilled, &cell_steps);
        __syncthreads();
        RAY_STAMP(2);

        // ---- in-place write-back. A window row is at most 34 groups of 8 cells (one 128-bit shared load each); a
        // non-empty group is two 128-bit global read-modify-writes. Main pass: one warp per row, lane g
        // takes group g < 32, RAY_WB_ROWS rows in flight per warp. Tail pass: the (at most two) groups
        // beyond the 32nd of each row, one thread per row.
        const uint4* win4 = reinterpret_cast<const uint4*>(s_win);
        constexpr int RAY_WB_ROWS = 2;   // (measured on a configs[4] shard: 2 -> 0.770 ms per step, 4 -> 0.800: four rows spilled)
        int exmin = 0x7fffffff, eymin = 0x7fffffff, exmax = -1, eymax = -1;   // this thread's touched extent
        for (int ly0 = warp; ly0 < wh; ly0 += n_warps * RAY_WB_ROWS) {
            uint4 d[RAY_WB_ROWS], va[RAY_WB_ROWS], vb[RAY_WB_ROWS];
            uint4* gp[RAY_WB_ROWS];
            bool nz[RAY_WB_ROWS];
#pragma unroll
            for (int j = 0; j < RAY_WB_ROWS; ++j) {
                const int ly = ly0 + j * n_warps;
                nz[j] = false;
                if (ly < wh) {
                    const int2 row = s_row[ly];
                    if (lane < (row.y >> 19)) {          // width / 8 groups in this row
                        d[j] = win4[(row.x >> 3) + lane];
                        nz[j] = (d[j].x | d[j].y | d[j].z | d[j].w) != 0u;
                        if (nz[j]) {
                            const int gx0 = (row.y & 0xffff) + 8 * lane;
                            exmin = min(exmin, gx0); exmax = max(exmax, gx0 + 7);
                            eymin = min(eymin, wy0 + ly); eymax = max(eymax, wy0 + ly);
                            gp[j] = reinterpret_cast<uint4*>(grid + phys_index(geom, (uint32_t)gx0, (uint32_t)(wy0 + ly)));
                        }
                    }
                }
            }
#pragma unroll
            for (int j = 0; j < RAY_WB_ROWS; ++j)
                if (nz[j]) ld_group_v8(gp[j], va[j], vb[j]);
#pragma unroll
            for (int j = 0; j < RAY_WB_ROWS; ++j) {   // band extent of the row: first / last non-empty group
                const unsigned mnz = __ballot_sync(0xffffffffu, nz[j]);
                const int ly = ly0 + j * n_warps;
                if (mnz != 0u && lane == 0) {
                    const int rx0 = s_row[ly].y & 0xffff;
                    band_add(s_blo, s_bhi, band0, wy0 + ly, rx0 + 8 * (__ffs(mnz) - 1), rx0 + 8 * (31 - __clz(mnz)) + 7);
                }
            }
#pragma unroll
            for (int j = 0; j < RAY_WB_ROWS; ++j) {
                if (nz[j]) {
                    merge_window_group(va[j], vb[j], d[j], &saturated);
                    st_group_v8(gp[j], va[j], vb[j]);
                }
            }
        }
        for (int ly = threadIdx.x; ly < wh; ly += blockDim.x) {   // tail pass: groups 32, 33 of each row
            const int2 row = s_row[ly];
            for (int g = 32; g < (row.y >> 19); ++g) {
                const uint4 dd = win4[(row.x >> 3) + g];
                if ((dd.x | dd.y | dd.z | dd.w) == 0u) continue;
                const int gx0 = (row.y & 0xffff) + 8 * g;
                exmin = min(exmin, gx0); exmax = max(exmax, gx0 + 7);
                eymin = min(eymin, wy0 + ly); eymax = max(eymax, wy0 + ly);
                band_add(s_blo, s_bhi, band0, wy0 + ly, gx0, gx0 + 7);
                uint4* gpt = reinterpret_cast<uint4*>(grid + phys_index(geom, (uint32_t)gx0, (uint32_t)(wy0 + ly)));
                uint4 ta = gpt[0], tb = gpt[1];
                merge_window_group(ta, tb, dd, &saturated);
                gpt[0] = ta;
                gpt[1] = tb;
            }
        }
        ext_add(s_ext, exmin, eymin, exmax, eymax);
        __syncthreads();
        band_commit(s_blo, s_bhi, band0, bands, geom);
        if (threadIdx.x == 0) ext_commit(s_ext, &meta[slot], (int)geom.gw);
        RAY_STAMP(5);
#ifdef SLAMRS_RAY_TRACE
        if (threadIdx.x == 0) atomicAdd(&g_ray_trace_items[1], 1ull);
#endif
    }
    if (saturated) atomicAdd(&counters->saturated, 1ull);
    if (spilled) atomicAdd(&counters->spilled, (unsigned long long)spilled);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cell_steps += __shfl_down_sync(0xffffffffu, cell_steps, o);
    if ((threadIdx.x & 31) == 0 && cell_steps) atomicAdd(&counters->ray_cell_steps, (unsigned long long)cell_steps);
}

// =============================================================================== k_ray_update_half
// The packed ray update with HALF a particle per work item (whole-grid tiled slots). A particle's rays
// either never leave the rows at or above its start row (y_inc >= 0: the "upper" half) or never leave the
// rows at or below it (y_inc < 0: the "lower" half), so each half needs only half the disc window
// (<= 54 KB at a 6 m / 5 cm window): four CTAs of 192 threads per SM instead of two of 384, 592 resident
// work slots instead of 296. With ~450 survivors per step the full-item kernel ran two rounds, the
// second on a third of the machine; 900 half items on 592 slots finish in about one item time
// (profiles/r2_ray_half.md).
//
// Ownership. The lower half owns the rows below the start row, the upper half the start row and
// everything above: each copies / writes only rows it owns, so the two CTAs never touch the same cell.
// The one shared row is the start row, which every lower ray also crosses: the lower CTA hands its
// window row for it to the upper CTA through a small exchange record (plus what the upper half needs to
// write the extent of the band both halves share), and the upper CTA adds it when it writes that row.
// The lower half is listed right before the upper half, so the upper CTA only ever waits for a CTA that
// is already running.
//
// Fused copies (deferred copies). A surviving particle whose grid is still an alias of its source's slot
// ("clone") would first need its own copy of the source's cells (k_copy_boxed) and then read them again to
// add the scan. Here its CTAs do both in one pass: one write-back path for clones and owners reads the ROOT
// slot's tiles (a clone's source; an owner's own slot), adds the window and writes the particle's OWN slot
// (and clears what the slot's previous tenant had informed outside the new extent). The copy kernels and
// their pass over the grids disappear from the step. The hazard is the root's owner integrating the scan in
// place while a clone still reads the root: k_resample_indices lists the clones first and the particles that
// own their slot after them and counts the readers of each root (readers[]; each half of a clone is one),
// every clone half announces when it has read its root (done[]), and an owner waits for its readers before it
// writes. Items are popped in list order by CTAs that are all resident, so every reader an owner waits for is
// already running: no deadlock.
constexpr int HALF_MAX_ROWS = RAY_MAX_RADIUS + 1;
constexpr int HALF_MAX_BANDS = HALF_MAX_ROWS / BAND_ROWS + 2;
constexpr uint32_t HALF_XCHG_GROUPS = 36;
struct alignas(16) HalfXchg {           // lower half -> upper half of the same particle
    uint4 row[HALF_XCHG_GROUPS];        // the lower CTA's window row for the start row (packed 16-bit cells, 8 per group)
    int band_lo, band_hi;               // columns the lower half touched in its rows of the shared band (hi < lo: none)
    uint32_t n_hits;                    // parked hits of lower rays on the start row (applied by the upper CTA)
    uint32_t pad;
    int ext[4];                         // what the lower half touched {xmin, ymin, xmax, ymax} (the upper half commits the slot's box)
    uint4 occ[HALF_XCHG_GROUPS];        // those hits: occupied count per start-row window cell (16 bits, cells as in `row`)
};
static_assert(sizeof(HalfXchg) % 16 == 0, "exchange records are accessed as 16-byte pieces");

// cells of the half-disc window of radius `radius`: rows start and end on multiples of 8 columns, so the size
// depends on the start column modulo 8 -- the largest of the eight cases (clipping at the grid only shrinks it)
__host__ __device__ inline int ray_window_cells_upper_bound_half(int radius) {
    int worst = 0;
    for (int a = 0; a < 8; ++a) {
        int total = 0;
        for (int dy = 0; dy <= radius; ++dy) {
            const int hw = isqrt_small(radius * radius - dy * dy), cx = 4096 + a;
            total += ((cx + hw + 1 + 7) & ~7) - ((cx - hw) & ~7);
        }
        worst = total > worst ? total : worst;
    }
    return worst;
}

// write-back of one half item: root tiles + window -> own slot, for the rows this half owns
__device__ __noinline__ void ray_half_writeback(const MapGeom& geom, const RayItem& it, bool upper, int cy0, bool walked,
                                                uint32_t* __restrict__ cells, SlotMeta* __restrict__ meta,
                                                uint32_t* __restrict__ bands_all, size_t cells_per_grid, const uint32_t* s_win,
                                                const int2* s_row, int* s_blo, int* s_bhi, int* s_ext, const uint4* s_lrow,
                                                const int* s_xinfo /* lower half's band range, valid for the upper half */,
                                                uint32_t eo_shared, int wy0, int wh, int band0, bool* saturated_p,
                                                uint32_t* moved_p) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, n_warps = blockDim.x >> 5;
    const uint32_t n_bands_slot = bands_per_slot(geom);
    const bool fused = it.root != it.slot;
    uint32_t* grid = cells + (size_t)it.slot * cells_per_grid;
    uint32_t* bands = bands_all + (size_t)it.slot * n_bands_slot;
    const uint32_t* src = cells + (size_t)it.root * cells_per_grid;
    const uint32_t* src_bands = bands_all + (size_t)it.root * n_bands_slot;
    bool saturated = false;
    uint32_t moved = 0;
    const uint4* win4 = reinterpret_cast<const uint4*>(s_win);
    // rows this half owns: the lower half everything below the start row, the upper half the rest
    const int own_lo = upper ? cy0 : 0, own_hi = upper ? (int)geom.gh : cy0;     // [own_lo, own_hi)
    if (own_hi <= own_lo) { *moved_p += 0; return; }
    const int shared_band = (cy0 % BAND_ROWS) ? cy0 / BAND_ROWS : -1;            // the band both halves have rows in
    // bands to visit: the source's rows, the rows the slot's previous tenant had informed, the touched rows -- clipped to the owned rows
    const SlotMeta sm = meta[it.root];
    int y_lo = 0x7fffffff, y_hi = -1;                                             // rows [y_lo, y_hi]
    if (sm.x1 > sm.x0 && sm.y1 > sm.y0) { y_lo = min(y_lo, sm.y0); y_hi = max(y_hi, sm.y1 - 1); }
    if (fused && it.old_y1 > it.old_y0) { y_lo = min(y_lo, it.old_y0); y_hi = max(y_hi, it.old_y1 - 1); }
    if (s_ext[3] >= s_ext[1] && s_ext[2] >= s_ext[0]) { y_lo = min(y_lo, s_ext[1]); y_hi = max(y_hi, s_ext[3]); }
    y_lo = max(y_lo, own_lo); y_hi = min(y_hi, own_hi - 1);
    if (y_hi < y_lo) { return; }
    const int by0 = y_lo / BAND_ROWS, by1 = y_hi / BAND_ROWS;
    const uint32_t tpr = geom.tiles_per_row;
    constexpr int DEPTH = 2;                   // tiles in flight per warp (measured: 2 -> 97 us per launch, 3 -> 98, 4 -> 104, 6 -> 136 with spills)
    const int rr = lane >> 2, uu = lane & 3;   // this lane's row of the band and 32-byte unit of the tile row
    for (int bnd = by0 + warp; bnd <= by1; bnd += n_warps) {
        const bool is_shared = bnd == shared_band;
        const uint32_t es = src_bands[bnd];
        const uint32_t eo = fused ? ((is_shared && !upper) ? eo_shared : bands[bnd]) : es;
        const int lb = bnd - band0;
        bool touched = (unsigned)lb < (unsigned)HALF_MAX_BANDS && s_bhi[lb] >= s_blo[lb];
        uint32_t t0x = touched ? ((uint32_t)s_blo[lb] & ~7u) : 0xffffu, t1x = touched ? min(geom.gw, ((uint32_t)s_bhi[lb] + 8u) & ~7u) : 0u;
        // the entry of the shared band also covers what the lower half touched in its rows of it
        uint32_t n0 = t0x, n1 = t1x;
        if (is_shared && upper && s_xinfo[1] >= s_xinfo[0]) { n0 = min(n0, (uint32_t)s_xinfo[0] & ~7u); n1 = max(n1, min(geom.gw, ((uint32_t)s_xinfo[1] + 8u) & ~7u)); }
        if (es) { n0 = min(n0, es & 0xffffu); n1 = max(n1, es >> 16); }
        // columns to write: a clone's rows get the source's cells and lose the previous tenant's; an owner's only change where hit
        uint32_t u0 = t0x, u1 = t1x;
        if (fused) { if (es) { u0 = min(u0, es & 0xffffu); u1 = max(u1, es >> 16); } if (eo) { u0 = min(u0, eo & 0xffffu); u1 = max(u1, eo >> 16); } }
        __syncwarp();                                   // every lane has read the old entry
        if (lane == 0 && (upper || !is_shared)) bands[bnd] = n1 > n0 ? (n0 | (n1 << 16)) : 0u;   // (the upper half writes the shared band's)
        if (u1 <= u0) continue;
        const int t_lo = (int)(u0 / TILE_COLS), t_hi = (int)((u1 + TILE_COLS - 1u) / TILE_COLS);
        const int y = bnd * BAND_ROWS + rr, ly = y - wy0;
        const bool own_row = y >= own_lo && y < own_hi;
        int wfirst = 0, wx0 = 0, ww = 0;
        if (walked && touched && (unsigned)ly < (unsigned)wh) { const int2 row = s_row[ly]; wfirst = row.x; wx0 = row.y & 0xffff; ww = row.y >> 16; }
        const bool start_row = upper && walked && y == cy0;                         // also receives the lower half's window row
        const uint32_t sx0 = es & 0xffffu, sx1 = es >> 16;                           // (0, 0 when the source has nothing here)
        const size_t band_off = (size_t)bnd * tpr * TILE_CELLS + 8u * (uint32_t)lane;
        for (int tt = t_lo; tt < t_hi; tt += DEPTH) {
            uint4 va[DEPTH], vb[DEPTH], d[DEPTH];
            bool need[DEPTH];
#pragma unroll
            for (int k = 0; k < DEPTH; ++k) {         // what the window adds to this lane's 8 cells of tile tt + k
                const int t = tt + k;
                const int lx = t * (int)TILE_COLS + 8 * uu - wx0;
                d[k] = make_uint4(0u, 0u, 0u, 0u);
                bool lower_too = false;
                if (t < t_hi && own_row && (unsigned)lx < (unsigned)ww) {
                    d[k] = win4[(wfirst + lx) >> 3];
                    if (start_row && (uint32_t)(lx >> 3) < HALF_XCHG_GROUPS) {
                        const uint4 dl = s_lrow[lx >> 3];
                        lower_too = (dl.x | dl.y | dl.z | dl.w) != 0u;
                    }
                }
                // a clone's rows are written everywhere (copy + clear); an owner's only where something was hit
                need[k] = t < t_hi && own_row && (fused || lower_too || (d[k].x | d[k].y | d[k].z | d[k].w) != 0u);
            }
#pragma unroll
            for (int k = 0; k < DEPTH; ++k) {
                const int t = tt + k;
                const uint32_t x = (uint32_t)t * TILE_COLS + 8u * (uint32_t)uu;
                va[k] = make_uint4(0u, 0u, 0u, 0u); vb[k] = va[k];
                if (need[k] && x >= sx0 && x < sx1) {
                    const V8 s8 = ld_stream_v8(reinterpret_cast<const V8*>(src + band_off + (size_t)t * TILE_CELLS));
                    va[k] = s8.a; vb[k] = s8.b;
                    moved += fused ? 1u : 0u;   // (clone copies only: an owner's read-modify-write is the ray update's own traffic)
                }
            }
#pragma unroll
            for (int k = 0; k < DEPTH; ++k) {
                if (!need[k]) continue;
                const int t = tt + k;
                if ((d[k].x | d[k].y | d[k].z | d[k].w) != 0u) merge_window_group(va[k], vb[k], d[k], &saturated);
                if (start_row) {
                    const int lx = t * (int)TILE_COLS + 8 * uu - wx0;
                    if ((unsigned)lx < (unsigned)ww && (uint32_t)(lx >> 3) < HALF_XCHG_GROUPS) {
                        const uint4 dl = s_lrow[lx >> 3];
                        if ((dl.x | dl.y | dl.z | dl.w) != 0u) merge_window_group(va[k], vb[k], dl, &saturated);
                    }
                }
                V8 o8; o8.a = va[k]; o8.b = vb[k];
                st_stream_v8(reinterpret_cast<V8*>(grid + band_off + (size_t)t * TILE_CELLS), o8);
                moved += fused ? 1u : 0u;   // (clone copies only: an owner's read-modify-write is the ray update's own traffic)
            }
        }
    }
    if (saturated) *saturated_p = true;
    *moved_p += moved;
}

__global__ void __maxnreg__(80)   // 4 CTAs of 192 threads per SM
k_ray_update_half(MapGeom geom, ScanDevice scan, const ParticleResult* __restrict__ results, uint32_t first_particle,
                  const uint32_t* __restrict__ alive_list, const RayItem* __restrict__ clones, const RayItem* __restrict__ owners,
                  const uint32_t* __restrict__ readers, uint32_t* __restrict__ done, uint32_t* __restrict__ xflag,
                  HalfXchg* __restrict__ xchg, uint32_t* __restrict__ spill_scratch, const int32_t* __restrict__ slot_of,
                  uint32_t* __restrict__ cells, SlotMeta* __restrict__ meta, uint32_t* __restrict__ bands_all,
                  size_t cells_per_grid, int radius, uint32_t window_bytes, StepCounters* counters,
                  uint32_t* __restrict__ xdone, uint32_t n_local, uint32_t signal_epoch) {
    extern __shared__ __align__(16) uint32_t s_win[];   // two 16-bit cells per word; behind the window: this half's beam list
    uint16_t* s_beam = reinterpret_cast<uint16_t*>(reinterpret_cast<unsigned char*>(s_win) + window_bytes);
    __shared__ uint32_t s_nspill, s_nmine, s_eo_shared, s_nxhits;
    __shared__ int s_blo[HALF_MAX_BANDS], s_bhi[HALF_MAX_BANDS];
    __shared__ int2 s_row[HALF_MAX_ROWS + 1];           // .x = first window cell of the row, .y = x0 | width << 16
    __shared__ uint32_t s_rowb[HALF_MAX_ROWS];          // shared byte address of column x = 0 of the row
    __shared__ int s_ext[4], s_xinfo[2], s_lext[4];
    __shared__ unsigned long long s_next;
    __shared__ RayItem s_item;                          // the item s_next names and its particle's pose, fetched ahead
    __shared__ float s_pose[3];
    __shared__ uint4 s_lrow[HALF_XCHG_GROUPS];
    const unsigned long long n_items = counters->n_alive;
    const int gw = (int)geom.gw, gh = (int)geom.gh;
    const uint32_t win_base = (uint32_t)__cvta_generic_to_shared(s_win);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, n_warps = blockDim.x >> 5;
    const uint32_t n_bands_slot = bands_per_slot(geom);
    bool saturated = false;
    uint32_t spilled = 0, cell_steps = 0, moved = 0;
    uint32_t* my_spill = spill_scratch + (size_t)blockIdx.x * RAY_SPILL_CAP;
    // Global round trips that nothing in the item waits for are taken by one lane of the last warp (the shortest
    // beams) while the CTA walks: popping the NEXT work item, and the previous item's box commit and "root has
    // been read" signal.
    const bool helper = threadIdx.x == blockDim.x - 32u;
    SlotMeta* pend_meta = nullptr;      // helper lane: box of the previous item to union `pend_ext` into
    uint32_t* pend_done = nullptr;      // helper lane: reader counter to bump for the previous item
    int pend_ext[4] = {0, 0, -1, -1};
    // world > 1 (signal_epoch != 0): a peer GPU that pulls this slot in this step waits for `signal_epoch` in the
    // slot's SlotMeta::pad0. The half that finishes second publishes it, after the box commit.
    uint32_t* pend_sig = nullptr;       // helper lane: xdone counter of the previous item
    SlotMeta* pend_sig_meta = nullptr;
    auto flush_pending = [&]() {
        if (pend_meta != nullptr) {
            SlotMeta b = *pend_meta;
            const int am = BOX_ALIGN - 1;
            const int x0 = pend_ext[0] & ~am, x1 = min(gw, (pend_ext[2] + 1 + am) & ~am), y0 = pend_ext[1], y1 = pend_ext[3] + 1;
            if (b.x1 <= b.x0) { b.x0 = x0; b.y0 = y0; b.x1 = x1; b.y1 = y1; }
            else { b.x0 = min(b.x0, x0); b.y0 = min(b.y0, y0); b.x1 = max(b.x1, x1); b.y1 = max(b.y1, y1); }
            *pend_meta = b;
            pend_meta = nullptr;
        }
        if (pend_done != nullptr) {
            __threadfence();
            atomicAdd(pend_done, 1u);        // that half has read the root: its owner may write it
            pend_done = nullptr;
        }
        if (pend_sig != nullptr) {
            __threadfence_system();          // this half's cells, band entries and (upper half) the box
            if (atomicAdd(pend_sig, 1u) == 1u) {   // the other half was first: everything of this slot is in place
                __threadfence_system();
                asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(&pend_sig_meta->pad0), "r"(signal_epoch) : "memory");
            }
            pend_sig = nullptr;
        }
    };
    // pops the next work item and fetches what every thread needs of it (one thread, while the others walk)
    auto pop_next = [&]() {
        const unsigned long long w = atomicAdd(&counters->ray_work_head, 1ull);
        if (w < 2ull * n_items) {
            RayItem nit;
            if (clones) nit = ray_item_at(clones, owners, n_local, counters, w >> 1);   // clones first: an owner is popped only after every clone that reads its slot
            else { nit.particle = alive_list[w >> 1]; nit.slot = slot_of[nit.particle]; nit.root = nit.slot; nit.old_y0 = nit.old_y1 = 0; nit.pad = 0u; }
            const ParticleResult r = results[first_particle + nit.particle];
            s_item = nit;
            s_pose[0] = r.x; s_pose[1] = r.y; s_pose[2] = r.theta;
        }
        s_next = w;
    };
    if (threadIdx.x == 0) pop_next();
#ifdef SLAMRS_RAY_TRACE
    long long t_prev = clock64();
#endif

    for (;;) {
        __syncthreads();       // the previous item's shared state is no longer read; s_next holds this item
        const unsigned long long work = s_next;
        if (work >= 2ull * n_items) break;
        RAY_STAMP(0);
        RAY_LOG(work, 0);
        const unsigned long long item = work >> 1;
        const bool upper = (work & 1ull) != 0ull;   // the lower half of a particle is listed first
        const RayItem it = s_item;
        const bool fused = it.root != it.slot;
        uint32_t* grid = cells + (size_t)it.slot * cells_per_grid;
        uint32_t* bands = bands_all + (size_t)it.slot * n_bands_slot;
        const float px = s_pose[0], py = s_pose[1], ptheta = s_pose[2];
        const float sx = world_to_grid(px, geom.pos_x, geom.res);
        const float sy = world_to_grid(py, geom.pos_y, geom.res);
        const long long lcx = f32_as_isize(floorf(sx)), lcy = f32_as_isize(floorf(sy));
        // every ray starts in the same cell; outside the grid nothing is emitted (ray.rs:88-92)
        const bool walked = !(lcx < 0 || lcx >= (long long)geom.gw || lcy < 0 || lcy >= (long long)geom.gh);
        if (!walked && !fused) {   // nothing to do (both halves agree); the next item still has to be popped
            __syncthreads();
            if (helper) {
                flush_pending();
                pop_next();
                if (signal_epoch != 0u && it.pad != 0u) { pend_sig = xdone + item; pend_sig_meta = &meta[it.slot]; }
            }
            continue;
        }
        // (a clone whose pose left the grid integrates nothing but still gets its own cells: the upper half copies all rows)
        const int cx0 = walked ? (int)lcx : 0, cy0 = walked ? (int)lcy : 0;
        const int rad = walked ? radius : 0;
        ext_init(s_ext);
        if (threadIdx.x == 0) {
            s_nspill = 0u; s_nmine = 0u; s_xinfo[0] = 0x7fffffff; s_xinfo[1] = -1; s_eo_shared = 0u; s_nxhits = 0u;
            s_lext[0] = s_lext[1] = 0x7fffffff; s_lext[2] = s_lext[3] = -1;
        }
        for (int i = threadIdx.x; i < HALF_MAX_BANDS; i += blockDim.x) { s_blo[i] = 0x7fffffff; s_bhi[i] = -1; }
        if (threadIdx.x < HALF_XCHG_GROUPS) s_lrow[threadIdx.x] = make_uint4(0u, 0u, 0u, 0u);

        // ---- row table of the half-disc window (x ranges aligned to 8 cells = one 128-bit group)
        const int wy0 = upper ? cy0 : max(0, cy0 - rad), wy1 = upper ? min(gh, cy0 + rad + 1) : cy0 + 1;
        const int band0 = wy0 / BAND_ROWS;
        const int wh = walked ? wy1 - wy0 : 0;
        for (int ly = threadIdx.x; ly < wh; ly += blockDim.x) {
            const int dy = wy0 + ly - cy0;
            const int hw = isqrt_small(rad * rad - dy * dy);
            const int x0 = max(0, cx0 - hw) & ~7;
            const int x1 = min(gw, (min(gw, cx0 + hw + 1) + 7) & ~7);
            s_row[ly].y = x0 | ((x1 - x0) << 16);
        }
        __syncthreads();
        if (threadIdx.x >= 32) {   // the other warps clear the window while warp 0 lays out its rows
            uint4* w4 = reinterpret_cast<uint4*>(s_win);
            for (int i = threadIdx.x - 32; i < (int)(window_bytes >> 4); i += blockDim.x - 32) w4[i] = make_uint4(0u, 0u, 0u, 0u);
        }
        if (threadIdx.x < 32) {
            int carry = 0;
            for (int base = 0; base < wh; base += 32) {
                const int ly = base + (int)threadIdx.x;
                const int w = ly < wh ? (s_row[ly].y >> 16) : 0;
                int inc = w;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const int t = __shfl_up_sync(0xffffffffu, inc, o);
                    if ((int)threadIdx.x >= o) inc += t;
                }
                if (ly < wh) {
                    const int first = carry + inc - w;
                    s_row[ly].x = first;
                    s_rowb[ly] = win_base + 2u * (uint32_t)(first - (s_row[ly].y & 0xffff));
                }
                carry += __shfl_sync(0xffffffffu, inc, 31);
            }
            if (threadIdx.x == 0) s_row[wh] = make_int2(carry, 0);
        }
        __syncthreads();
        RAY_STAMP(1);
        RAY_LOG(work, 1);
        // ---- which beams are this half's: y_inc >= 0 (upper) or < 0 (lower), decided exactly as the iterator does
        //      (ray.rs:54-72); a cheap test settles all but the nearly horizontal ones
        if (walked) {
            for (uint32_t t0 = 0; t0 < scan.n_beams; t0 += blockDim.x) {
                const uint32_t t = t0 + threadIdx.x;
                bool mine = false;
                uint32_t b = 0u;
                if (t < scan.n_beams) {
                    b = scan.order ? scan.order[t] : t;
                    const float dist = scan.dist[b];
                    const float a = __fadd_rn(ptheta, scan.angle[b]);
                    const float dyq = __fmul_rn(sinf(a), dist);
                    const float margin = 1.0e-4f * (fabsf(py) + fabsf(geom.pos_y) + fabsf(dist) + geom.res);
                    bool up;
                    if (dyq > margin) up = true;
                    else if (dyq < -margin) up = false;
                    else {
                        float ex, ey;
                        beam_endpoint(px, py, ptheta, scan.angle[b], dist, &ex, &ey);
                        const float y1 = world_to_grid(ey, geom.pos_y, geom.res);
                        up = fabsf(__fsub_rn(y1, sy)) == 0.0f || y1 > sy;
                    }
                    mine = up == upper;
                }
                const unsigned m = __ballot_sync(0xffffffffu, mine);
                if (m) {
                    uint32_t base = 0u;
                    if (lane == 0) base = atomicAdd(&s_nmine, (uint32_t)__popc(m));
                    base = __shfl_sync(0xffffffffu, base, 0);
                    if (mine) s_beam[base + __popc(m & ((1u << lane) - 1u))] = (uint16_t)b;
                }
            }
        }
        __syncthreads();
        RAY_STAMP(2);
        RAY_LOG(work, 2);
        if (helper) {
            flush_pending();
            pop_next();   // (s_next, s_item, s_pose are read only after the barrier that ends this item)
        }
        if (walked) {
            // the window holds every in-grid cell within `rad` of the start in this half's rows
            const bool disc_in_grid = cx0 - rad >= 0 && cx0 + rad < gw && (upper ? cy0 + rad < gh : cy0 - rad >= 0);
            ray_walk_packed<true>(geom, scan, s_beam, s_nmine, px, py, ptheta, sx, sy, cx0, cy0, rad, disc_in_grid, wy0, wh, band0,
                                  s_win, s_row, s_rowb, s_blo, s_bhi, s_ext, nullptr, nullptr, &s_nspill, my_spill, nullptr,
                                  &spilled, &cell_steps);
        }
#ifdef SLAMRS_RAY_TRACE
        if (threadIdx.x == 0) atomicAdd(&g_ray_trace[12], (unsigned long long)(clock64() - t_prev));   // warp 0's own walk (longest beams)
#endif
        __syncthreads();
        RAY_STAMP(3);
        RAY_LOG(work, 3);

        // ---- per band of the window the columns that really received hits (a lane scans one window row; the lower
        //      half leaves the start row to the upper half)
        const uint4* win4 = reinterpret_cast<const uint4*>(s_win);
        {
            const int rr = lane & 7, bq = lane >> 3;
            int wxmin = 0x7fffffff, wymin = 0x7fffffff, wxmax = -1, wymax = -1;
            const int n_wbands = wh > 0 ? (wy0 + wh - 1) / BAND_ROWS - band0 + 1 : 0;
            for (int q = warp; 4 * q < n_wbands; q += n_warps) {
                const int lb = 4 * q + bq;
                const int y = (band0 + lb) * BAND_ROWS + rr, ly = y - wy0;
                int first = 0x7fffffff, last = -1, rx0 = 0;
                int2 row = make_int2(0, 0);
                if (lb < n_wbands && (unsigned)ly < (unsigned)wh && (upper || y != cy0)) { row = s_row[ly]; rx0 = row.y & 0xffff; }
                const int groups = row.y >> 19;
                for (int g = 0; g < 34; ++g) {                 // (a window row is at most 34 groups wide)
                    if (__all_sync(0xffffffffu, g >= groups)) break;
                    if (g < groups) {
                        const uint4 d = win4[(row.x >> 3) + g];
                        if ((d.x | d.y | d.z | d.w) != 0u) { first = min(first, g); last = g; }
                    }
                }
                int xlo = last >= 0 ? rx0 + 8 * first : 0x7fffffff, xhi = last >= 0 ? rx0 + 8 * last + 7 : -1;
                if (last >= 0) { wymin = min(wymin, y); wymax = max(wymax, y); }
#pragma unroll
                for (int o = 1; o < 8; o <<= 1) {
                    xlo = min(xlo, __shfl_xor_sync(0xffffffffu, xlo, o));
                    xhi = max(xhi, __shfl_xor_sync(0xffffffffu, xhi, o));
                }
                wxmin = min(wxmin, xlo); wxmax = max(wxmax, xhi);
                if (rr == 0 && xhi >= xlo && (unsigned)lb < (unsigned)HALF_MAX_BANDS) { atomicMin(&s_blo[lb], xlo); atomicMax(&s_bhi[lb], xhi); }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                wxmin = min(wxmin, __shfl_xor_sync(0xffffffffu, wxmin, o)); wxmax = max(wxmax, __shfl_xor_sync(0xffffffffu, wxmax, o));
                wymin = min(wymin, __shfl_xor_sync(0xffffffffu, wymin, o)); wymax = max(wymax, __shfl_xor_sync(0xffffffffu, wymax, o));
            }
            if (lane == 0) ext_add(s_ext, wxmin, wymin, wxmax, wymax);
        }
        __syncthreads();
        RAY_STAMP(4);
        RAY_LOG(work, 4);

        // ---- the start row is shared: the lower half hands its window row for it (and what the upper half needs
        //      for the band both halves have rows in) to the upper half
        const int shared_band = (cy0 % BAND_ROWS) ? cy0 / BAND_ROWS : -1;
        if (walked && !upper) {
            HalfXchg* x = xchg + item;
            const int2 row = s_row[wh - 1];                        // the start row is this window's last
            const int groups = row.y >> 19;
            // parked hits of lower rays on the start row travel too (the upper half writes that row), as 16-bit
            // counts per cell in s_lrow, which the lower half does not use otherwise
            {
                uint32_t* s_occ = reinterpret_cast<uint32_t*>(s_lrow);
                const uint32_t rx0 = (uint32_t)(row.y & 0xffff), ns = min(s_nspill, RAY_SPILL_CAP);
                for (uint32_t k = threadIdx.x; k < ns; k += blockDim.x) {
                    const uint32_t e = my_spill[k];
                    if ((int)((e >> 15) & 0x7fffu) != cy0) continue;
                    const uint32_t lx = (e & 0x7fffu) - rx0;
                    if ((e & 0x40000000u) && lx < 8u * HALF_XCHG_GROUPS) {
                        atomicAdd(&s_occ[lx >> 1], 1u << ((lx & 1u) << 4));
                        atomicAdd(&s_nxhits, 1u);
                    } else {
                        atomicAdd(&counters->fuse_overflow, 1ull);   // (a lower ray parks only occupied hits of window cells)
                    }
                }
            }
            __syncthreads();
            if (threadIdx.x < HALF_XCHG_GROUPS) {
                x->row[threadIdx.x] = (int)threadIdx.x < groups ? win4[(row.x >> 3) + threadIdx.x] : make_uint4(0u, 0u, 0u, 0u);
                x->occ[threadIdx.x] = s_lrow[threadIdx.x];
            }
            if (threadIdx.x == 0) {
                const int lb = shared_band - band0;
                const bool any = shared_band >= 0 && (unsigned)lb < (unsigned)HALF_MAX_BANDS && s_bhi[lb] >= s_blo[lb];
                x->band_lo = any ? s_blo[lb] : 0x7fffffff;
                x->band_hi = any ? s_bhi[lb] : -1;
                x->ext[0] = s_ext[0]; x->ext[1] = s_ext[1]; x->ext[2] = s_ext[2]; x->ext[3] = s_ext[3];
                x->n_hits = s_nxhits;
                // the shared band's old entry, before the upper half replaces it
                s_eo_shared = (fused && shared_band >= 0) ? bands[shared_band] : 0u;
            }
            __threadfence();
            __syncthreads();
            if (threadIdx.x == 0) asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(xflag + item), "r"(1u) : "memory");
        }
        if (walked && upper) {
            if (threadIdx.x == 0) {
                uint32_t seen;
                for (;;) {
                    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(xflag + item) : "memory");
                    if (seen != 0u) break;
                    __nanosleep(100);
                }
            }
            __syncthreads();
            const HalfXchg* x = xchg + item;
            if (threadIdx.x < HALF_XCHG_GROUPS) s_lrow[threadIdx.x] = __ldcg(&x->row[threadIdx.x]);
            if (threadIdx.x == 0) {
                s_xinfo[0] = __ldcg(&x->band_lo); s_xinfo[1] = __ldcg(&x->band_hi);
                s_lext[0] = __ldcg(&x->ext[0]); s_lext[1] = __ldcg(&x->ext[1]); s_lext[2] = __ldcg(&x->ext[2]); s_lext[3] = __ldcg(&x->ext[3]);
                s_nxhits = __ldcg(&x->n_hits);
            }
            __syncthreads();
            if (warp == 0) {   // what the lower rays touched on the start row counts for this half's extents
                const int2 row = s_row[0];
                const int rx0 = row.y & 0xffff;
                int first = 0x7fffffff, last = -1;
                for (int g = lane; g < (int)HALF_XCHG_GROUPS; g += 32) {
                    const uint4 d = s_lrow[g];
                    if ((d.x | d.y | d.z | d.w) != 0u) { first = min(first, g); last = max(last, g); }
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    first = min(first, __shfl_xor_sync(0xffffffffu, first, o));
                    last = max(last, __shfl_xor_sync(0xffffffffu, last, o));
                }
                if (lane == 0 && last >= 0) {
                    ext_add(s_ext, rx0 + 8 * first, cy0, rx0 + 8 * last + 7, cy0);
                    band_add(s_blo, s_bhi, band0, cy0, rx0 + 8 * first, rx0 + 8 * last + 7);
                }
            }
            __syncthreads();
        }
        RAY_STAMP(5);
        RAY_LOG(work, 5);
        // ---- an owner whose slot clones read in this step waits for them before it writes
        if (!fused && readers != nullptr) {
            if (threadIdx.x == 0) {
                const uint32_t want = readers[it.slot];
                if (want != 0u) {
                    uint32_t seen;
                    for (;;) {
                        asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(done + it.slot) : "memory");
                        if (seen >= want) break;
                        __nanosleep(100);
                    }
                }
            }
            __syncthreads();
        }
        RAY_STAMP(6);
        RAY_LOG(work, 6);
        ray_half_writeback(geom, it, upper, cy0, walked, cells, meta, bands_all, cells_per_grid, s_win, s_row, s_blo, s_bhi, s_ext,
                           s_lrow, s_xinfo, s_eo_shared, wy0, wh, band0, &saturated, &moved);
#ifdef SLAMRS_RAY_TRACE
        if (threadIdx.x == 0) atomicAdd(&g_ray_trace[13], (unsigned long long)(clock64() - t_prev));   // warp 0's own write-back
#endif
        __syncthreads();
        RAY_STAMP(fused ? 7 : 11);
        RAY_LOG(work, 7);
        RAY_LOG_V(work, 9, (unsigned long long)ray_smid() | ((unsigned long long)blockIdx.x << 16) | (fused ? 1ull << 40 : 0ull) | (upper ? 1ull << 41 : 0ull) | (it.pad ? 1ull << 42 : 0ull) | ((unsigned long long)s_nmine << 44));
#ifdef SLAMRS_RAY_TRACE
        if (threadIdx.x == 0) atomicAdd(&g_ray_trace_items[fused ? 0 : 1], 1ull);
#endif
        {   // the parked exact-path hits, now that the slot holds its cells (the lower half's start-row hits went to the upper half)
            const uint32_t ns = s_nspill;
            if (ns > RAY_SPILL_CAP && threadIdx.x == 0) atomicAdd(&counters->fuse_overflow, 1ull);
            for (uint32_t k = threadIdx.x; k < min(ns, RAY_SPILL_CAP); k += blockDim.x) {
                const uint32_t e = my_spill[k];
                const uint32_t x = e & 0x7fffu, y = (e >> 15) & 0x7fffu;
                if (!upper && (int)y == cy0) continue;
                global_cell_add(&grid[phys_index(geom, x, y)], (e & 0x40000000u) ? CELL_OCC_INC : CELL_FREE_INC, &saturated);
            }
            if (upper && walked && s_nxhits != 0u) {   // and the lower half's, n hits of a cell in one saturating add
                const uint32_t* occ = reinterpret_cast<const uint32_t*>(xchg[item].occ);
                const uint32_t rx0 = (uint32_t)(s_row[0].y & 0xffff);
                for (uint32_t k = threadIdx.x; k < 8u * HALF_XCHG_GROUPS; k += blockDim.x) {
                    const uint32_t n = (__ldcg(&occ[k >> 1]) >> ((k & 1u) << 4)) & 0xffffu;
                    if (n != 0u) global_cell_add(&grid[phys_index(geom, rx0 + k, (uint32_t)cy0)], n * CELL_OCC_INC, &saturated);
                }
            }
        }
        if (helper) {
            // The slot's box (a clone's was set to its source's when it was listed) grows by what both halves touched:
            // the upper half commits for both (the lower half's extent came with the exchange record), so the box has
            // one writer. Committed, like the reader signal, while the next item walks.
            if (upper && walked) {
                const int e0 = min(s_ext[0], s_lext[0]), e1 = min(s_ext[1], s_lext[1]), e2 = max(s_ext[2], s_lext[2]), e3 = max(s_ext[3], s_lext[3]);
                if (e2 >= e0 && e3 >= e1) { pend_meta = &meta[it.slot]; pend_ext[0] = e0; pend_ext[1] = e1; pend_ext[2] = e2; pend_ext[3] = e3; }
            }
            if (fused) pend_done = &done[it.root];
            if (signal_epoch != 0u && it.pad != 0u) { pend_sig = xdone + item; pend_sig_meta = &meta[it.slot]; }
        }
        RAY_STAMP(14);
        RAY_LOG(work, 8);
    }
    if (helper) flush_pending();
#ifdef SLAMRS_RAY_TRACE
    if (threadIdx.x == 0) { atomicAdd(&g_ray_trace[15], (unsigned long long)(clock64() - t_prev)); }
#endif
    if (saturated) atomicAdd(&counters->saturated, 1ull);
    if (spilled) atomicAdd(&counters->spilled, (unsigned long long)spilled);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { cell_steps += __shfl_down_sync(0xffffffffu, cell_steps, o); moved += __shfl_down_sync(0xffffffffu, moved, o); }
    if ((threadIdx.x & 31) == 0 && cell_steps) atomicAdd(&counters->ray_cell_steps, (unsigned long long)cell_steps);
    if ((threadIdx.x & 31) == 0 && moved) {
        atomicAdd(&counters->copy_bytes, (unsigned long long)moved * 32ull);
        atomicAdd(&counters->ray_copy_bytes, (unsigned long long)moved * 32ull);
    }
}

// =============================================================================== k_sort_beams
// Bitonic sort of (|dist|, beam index) in shared memory, descending; one CTA, once per scan, on the side
// stream while the likelihood kernel runs.
__global__ void __launch_bounds__(1024)
k_sort_beams(const float* __restrict__ dist, uint32_t n, uint16_t* __restrict__ order) {
    __shared__ float s_key[SORT_MAX_BEAMS];
    __shared__ uint16_t s_idx[SORT_MAX_BEAMS];
    for (uint32_t i = threadIdx.x; i < SORT_MAX_BEAMS; i += blockDim.x) {
        float k = -1.0f;                                    // padding and NaN sort last
        if (i < n) { const float d = fabsf(dist[i]); if (d == d) k = d; }
        s_key[i] = k;
        s_idx[i] = (uint16_t)i;
    }
    __syncthreads();
    for (uint32_t size = 2; size <= SORT_MAX_BEAMS; size <<= 1) {
        for (uint32_t stride = size >> 1; stride > 0; stride >>= 1) {
            for (uint32_t t = threadIdx.x; t < SORT_MAX_BEAMS / 2; t += blockDim.x) {
                const uint32_t lo = 2 * t - (t & (stride - 1));
                const uint32_t hi = lo + stride;
                const bool descending = (lo & size) == 0;
                const float a = s_key[lo], b = s_key[hi];
                // ties keep the lower beam index first: a total order, so the result is deterministic
                const bool a_first = a > b || (a == b && s_idx[lo] < s_idx[hi]);
                if (a_first != descending) {
                    s_key[lo] = b; s_key[hi] = a;
                    const uint16_t ti = s_idx[lo]; s_idx[lo] = s_idx[hi]; s_idx[hi] = ti;
                }
            }
            __syncthreads();
        }
    }
    for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) order[i] = s_idx[i];   // the n real beams come first
}
void launch_sort_beams(cudaStream_t stream, const float* dist, uint32_t n_beams, uint16_t* order) {
    k_sort_beams<<<1, 1024, 0, stream>>>(dist, n_beams, order);
}

static int ray_packed_radius(int radius_cells) {
    int radius = radius_cells < 1 ? 1 : (radius_cells > RAY_MAX_RADIUS ? RAY_MAX_RADIUS : radius_cells);
    while (radius > 1 && (size_t)ray_window_cells_upper_bound_packed(radius) * 2 > (size_t)RAY_MAX_SMEM) radius--;
    return radius;
}
// The fused path needs the packed kernel, whole-grid tiled slots (logical cell = physical cell) and a window
// that holds every cell a ray can reach (then only a 32nd occupied hit bypasses the window).
bool ray_update_can_fuse(const MapGeom& geom, uint32_t n_beams, size_t cells_per_grid, bool force_generic, int radius_cells) {
    return !force_generic && geom.gw % 8u == 0u && cells_per_grid % 8u == 0u && n_beams <= RAY_PACKED_MAX_BEAMS &&
           geom.tiled != 0u && geom.windowed == 0u && geom.gw < 32768u && geom.gh < 32768u &&
           ray_packed_radius(radius_cells) >= radius_cells;
}
#ifdef SLAMRS_RAY_TRACE
// tuning builds: after the SLAMRS_RAY_TRACE_LAUNCH-th launch of k_ray_update_half, dump its per-item timeline
static void ray_log_dump_after_launch(cudaStream_t stream) {
    static int launches = 0;
    const char* path = getenv("SLAMRS_RAY_TRACE_LOG");
    const char* which = getenv("SLAMRS_RAY_TRACE_LAUNCH");
    const int first = which ? atoi(which) : 20;
    ++launches;
    if (!path || launches < first || launches >= first + 4) return;
    int dev = 0;
    cudaGetDevice(&dev);
    const std::string name = std::string(path) + ".d" + std::to_string(dev) + "." + std::to_string(launches - first);
    path = name.c_str();
    cudaStreamSynchronize(stream);
    std::vector<unsigned long long> log((size_t)RAY_LOG_ITEMS * RAY_LOG_COLS);
    if (cudaMemcpyFromSymbol(log.data(), g_ray_log, log.size() * sizeof(unsigned long long)) == cudaSuccess) {
        if (FILE* f = fopen(path, "wb")) { fwrite(log.data(), sizeof(unsigned long long), log.size(), f); fclose(f); }
    }
}
#endif
int ray_trace(unsigned long long* out18) {
#ifdef SLAMRS_RAY_TRACE
    cudaError_t e = cudaMemcpyFromSymbol(out18, g_ray_trace, sizeof(unsigned long long) * 16);
    if (e == cudaSuccess) e = cudaMemcpyFromSymbol(out18 + 16, g_ray_trace_items, sizeof(unsigned long long) * 2);
    unsigned long long z[18] = {0};
    cudaMemcpyToSymbol(g_ray_trace, z, sizeof(unsigned long long) * 16);
    cudaMemcpyToSymbol(g_ray_trace_items, z, sizeof(unsigned long long) * 2);
    return (int)e;
#else
    (void)out18;
    return -1;
#endif
}
size_t ray_spill_scratch_words(int num_sms) { return (size_t)num_sms * 4u * RAY_SPILL_CAP; }   // <= 4 CTAs per SM

size_t ray_half_xchg_bytes() { return sizeof(HalfXchg); }

cudaError_t launch_ray_update(cudaStream_t stream, MapGeom geom, ScanDevice scan, const ParticleResult* results,
                              uint32_t first_particle, uint32_t n_local, const uint32_t* alive_list,
                              const RayItem* clones, const RayItem* owners, const uint32_t* readers, uint32_t* done,
                              uint32_t* xflag, void* xchg, uint32_t* spill_scratch, const int32_t* slot_of, uint32_t* cells,
                              SlotMeta* meta, uint32_t* bands, size_t cells_per_grid, int radius_cells, StepCounters* counters,
                              uint64_t* window_cells, bool force_generic, int num_sms, uint32_t* xdone, uint32_t signal_epoch) {
    // half a particle per work item (whole-grid tiled slots whose window holds every reachable cell): 4 CTAs per SM
    if (ray_update_can_fuse(geom, scan.n_beams, cells_per_grid, force_generic, radius_cells)) {
        const int radius = ray_packed_radius(radius_cells);
        const size_t wcells = (size_t)ray_window_cells_upper_bound_half(radius);
        const size_t wbytes = (wcells * 2 + 15) & ~(size_t)15;
        const size_t smem = wbytes + (((size_t)scan.n_beams * 2 + 15) & ~(size_t)15);
        int threads = (int)(((scan.n_beams + 1u) / 2u + 31u) / 32u * 32u) + 0;
        threads = threads < 128 ? 128 : (threads > RAY_MAX_THREADS ? RAY_MAX_THREADS : threads);
        *window_cells = 2 * wcells;
        int per_sm = 0;
        cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_ray_update_half, threads, smem);
        if (e != cudaSuccess) return e;
        if (per_sm < 1) per_sm = 1;
        if (per_sm > 4) per_sm = 4;   // (the spill scratch is sized for 4 CTAs per SM)
        uint32_t grid = (uint32_t)(per_sm * num_sms);
        if (grid > 2u * n_local) grid = 2u * n_local;
        k_ray_update_half<<<grid, threads, smem, stream>>>(geom, scan, results, first_particle, alive_list, clones, owners, readers, done,
                                                           xflag, (HalfXchg*)xchg, spill_scratch, slot_of, cells, meta, bands,
                                                           cells_per_grid, radius, (uint32_t)wbytes, counters, xdone, n_local, signal_epoch);
#ifdef SLAMRS_RAY_TRACE
        ray_log_dump_after_launch(stream);
#endif
        return cudaSuccess;
    }
    int threads = (int)((scan.n_beams + 31u) / 32u * 32u);
    threads = threads < 128 ? 128 : (threads > RAY_MAX_THREADS ? RAY_MAX_THREADS : threads);
    // the packed 16-bit window with a whole particle per CTA (two CTAs per SM at long range): row-major or windowed slots
    if (!force_generic && geom.gw % 8u == 0u && cells_per_grid % 8u == 0u && scan.n_beams <= RAY_PACKED_MAX_BEAMS) {
        const int radius = ray_packed_radius(radius_cells);
        const size_t wmax = (size_t)ray_window_cells_upper_bound_packed(radius);
        *window_cells = wmax;
        // as many CTAs as are resident at once, never more than there can be items
        int per_sm = 0;
        cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_ray_update_packed, threads, wmax * 2);
        if (e != cudaSuccess) return e;
        if (per_sm < 1) per_sm = 1;
        if (per_sm > 4) per_sm = 4;
        uint32_t grid = (uint32_t)(per_sm * num_sms);
        if (grid > n_local) grid = n_local;
        k_ray_update_packed<<<grid, threads, wmax * 2, stream>>>(geom, scan, results, first_particle, alive_list, slot_of, cells, meta,
                                                                 bands, cells_per_grid, radius, radius_cells, counters);
        return cudaSuccess;
    }
    const bool vec = (geom.gw % 4u == 0u) && (cells_per_grid % 4u == 0u);
    // largest disc radius whose row-aligned window fits the shared-memory budget
    int radius = radius_cells < 1 ? 1 : (radius_cells > RAY_MAX_RADIUS ? RAY_MAX_RADIUS : radius_cells);
    while (radius > 1 && (size_t)ray_window_cells_upper_bound(radius, vec) * 4 > (size_t)RAY_MAX_SMEM) radius--;
    const size_t wmax = (size_t)ray_window_cells_upper_bound(radius, vec);
    const size_t smem = wmax * 4;
    *window_cells = wmax;
    if (vec)
        k_ray_update<true><<<n_local, threads, smem, stream>>>(geom, scan, results, first_particle, alive_list, slot_of, cells, meta, bands,
                                                               cells_per_grid, radius, radius_cells, counters);
    else
        k_ray_update<false><<<n_local, threads, smem, stream>>>(geom, scan, results, first_particle, alive_list, slot_of, cells, meta, bands,
                                                                cells_per_grid, radius, radius_cells, counters);
    return cudaSuccess;
}

cudaError_t configure_ray_kernels() {
    // per-device opt-in to the large dynamic shared-memory window
    cudaError_t e = cudaFuncSetAttribute(k_ray_update<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, RAY_MAX_SMEM);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(k_ray_update_packed, cudaFuncAttributeMaxDynamicSharedMemorySize, RAY_MAX_SMEM);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(k_ray_update_half, cudaFuncAttributeMaxDynamicSharedMemorySize, RAY_MAX_SMEM / 2 + 8192);
    if (e != cudaSuccess) return e;
    return cudaFuncSetAttribute(k_ray_update<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, RAY_MAX_SMEM);
}

}  // namespace slamrs
