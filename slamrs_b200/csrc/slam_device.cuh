// Device-side arithmetic of the grid SLAM step. Every f32 operation that decides a cell index
// is an explicit round-to-nearest intrinsic so that nvcc can never contract a*b+c into an FMA
// (rustc does not contract); f32 division and sqrt are the IEEE-rounded forms.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "libm_f32.cuh"

namespace slamrs {

// ---------------------------------------------------------------------------- cell format
// One grid cell = packed hit counters: bits 0..15 = number of P_FREE updates, bits 16..31 =
// number of P_OCCUPPIED updates (P_PRIOR adds ln(1) = 0 and is dropped). The reference stores an
// f64 log-odds sum of the same three constants (slamrs/slam/src/grid/map.rs:154-156,
// common/src/math.rs:30-32), so the integer pair is an exact, order-independent encoding.
constexpr uint32_t CELL_FREE_INC = 1u;
constexpr uint32_t CELL_OCC_INC = 0x10000u;
// Probability(0.30).log_odds() and Probability(0.9).log_odds(), math.rs:30-32, in binary64
#define SLAMRS_L_FREE (-0.8472978603872036)
#define SLAMRS_L_OCC (2.1972245773362196)

__device__ __forceinline__ double cell_log_odds(uint32_t cell) {
    const double nf = (double)(cell & 0xffffu);
    const double no = (double)(cell >> 16);
    return __dadd_rn(__dmul_rn(nf, SLAMRS_L_FREE), __dmul_rn(no, SLAMRS_L_OCC));
}
// the scan matcher's occupancy test: log-odds > 0. No occupied hit means log-odds <= 0, so only cells with one read f64.
__device__ __forceinline__ bool cell_occupied(uint32_t cell) { return (cell >> 16) != 0u && cell_log_odds(cell) > 0.0; }
// LogOdds::probability, math.rs:135-137
__device__ __forceinline__ double log_odds_probability(double l) { return 1.0 - 1.0 / (1.0 + exp(l)); }

// one factor of Map::probability_of (map.rs:130-141) in log form for a cell of probability p:
// log(Z_HIT * p + (1 - Z_HIT) * 1 / SENSOR_MAXDIST), or log(1/1) when p is exactly the prior
__device__ __forceinline__ double beam_log_term_p(double prob) {
    // Z_HIT = 0.9, SENSOR_MAXDIST = 1.0 (map.rs:108-109)
    return (prob == 0.5) ? log(1.0 / 1.0) : log(__dadd_rn(__dmul_rn(0.9, prob), (1.0 - 0.9) * 1.0 / 1.0));
}
// the same for an informed cell given by its hit counters
__device__ __forceinline__ double beam_log_term(uint32_t cell) { return beam_log_term_p(log_odds_probability(cell_log_odds(cell))); }
// The factor depends on the cell's two hit counters only. For counters below these bounds it is
// read from a table that the same function filled on the same device at create (bit-identical
// to evaluating it in place, without the exp, the division and the log per beam).
constexpr uint32_t LK_TABLE_NF = 32, LK_TABLE_NO = 256;

__device__ __forceinline__ uint32_t cell_sat_add(uint32_t cell, uint32_t delta, bool* saturated) {
    uint32_t lo = (cell & 0xffffu) + (delta & 0xffffu);
    uint32_t hi = (cell >> 16) + (delta >> 16);
    if (lo > 0xffffu) { lo = 0xffffu; *saturated = true; }
    if (hi > 0xffffu) { hi = 0xffffu; *saturated = true; }
    return lo | (hi << 16);
}

// ---------------------------------------------------------------------------- Rust casts
// `f32 as usize` (saturating, NaN -> 0); only called for v >= 0 or NaN in the reference flow
__device__ __forceinline__ unsigned long long f32_as_usize(float v) {
    if (!(v == v)) return 0ull;
    if (v <= 0.0f) return 0ull;
    if (v >= 18446744073709551616.0f) return ~0ull;
    return (unsigned long long)v;
}
// `f32 as isize` (saturating, NaN -> 0)
__device__ __forceinline__ long long f32_as_isize(float v) {
    if (!(v == v)) return 0ll;
    if (v >= 9223372036854775808.0f) return 0x7fffffffffffffffll;
    if (v <= -9223372036854775808.0f) return (long long)0x8000000000000000ull;
    return (long long)v;
}

// ---------------------------------------------------------------------------- geometry
struct MapGeom {
    float pos_x, pos_y, res;
    uint32_t gw, gh;           // logical grid, cells
    // Physical slot. A slot stores logical cell (x, y) at row (y & ymask), column x & xmask.
    //  * Windowed slots (pw < gw or ph < gh, powers of two): a slot holds only a pw x ph torus of the
    //    logical grid. The mapping is injective on any extent that fits pw x ph, and a grid's informed
    //    extent is all a slot has to hold (everything else is the prior). Reads outside the extent
    //    return the prior without touching memory; an extent that would outgrow the window is an error
    //    (SLAMRS_E_WINDOW). This is what lets 32,768 particles with 2048 x 2048 maps share one B200.
    uint32_t pw, ph;           // slot width / height in cells (= gw, gh when not windowed)
    uint32_t xmask, ymask;
    uint32_t windowed;
    //  * Tiled slots (slot width a multiple of 32, height a multiple of 8): cells are stored tile by
    //    tile, a tile = 8 rows x 32 columns = 1 KiB = one DRAM page, tiles row-major. DRAM cost is per
    //    page touched, and the informed part of a band of 8 rows (~144 of 1024 columns) is 5 full tiles
    //    instead of 8 half-used row segments. The resampler copies whole tiles. (Row-major slots -- sides
    //    that are not multiples of 32 x 8 cells, e.g. the reference's 200^2 preset -- keep plain rows.)
    uint32_t tiled, tiles_per_row;
};
constexpr uint32_t TILE_COLS = 32, TILE_ROWS = 8, TILE_CELLS = TILE_COLS * TILE_ROWS;
__host__ __device__ inline bool is_pow2_u32(uint32_t v) { return v != 0u && (v & (v - 1u)) == 0u; }
// slot_cells = 0: a slot holds the whole grid; otherwise the slot is slot_cells x slot_cells (power of two)
__host__ __device__ inline MapGeom make_map_geom(float pos_x, float pos_y, float res, uint32_t gw, uint32_t gh,
                                                 uint32_t slot_cells = 0u) {
    MapGeom g;
    g.pos_x = pos_x; g.pos_y = pos_y; g.res = res; g.gw = gw; g.gh = gh;
    g.windowed = (slot_cells != 0u && (slot_cells < gw || slot_cells < gh)) ? 1u : 0u;
    g.pw = g.windowed ? (slot_cells < gw ? slot_cells : gw) : gw;
    g.ph = g.windowed ? (slot_cells < gh ? slot_cells : gh) : gh;
#ifndef SLAMRS_TILED
#define SLAMRS_TILED 1
#endif
    g.tiled = (SLAMRS_TILED && g.pw % TILE_COLS == 0u && g.ph % TILE_ROWS == 0u) ? 1u : 0u;
    g.tiles_per_row = g.pw / TILE_COLS;
    const bool ring = g.pw >= 256u && is_pow2_u32(g.pw);     // columns wrap (windowed slots)
    g.xmask = ring ? g.pw - 1u : 0xffffffffu;
    g.ymask = (g.windowed && is_pow2_u32(g.ph)) ? g.ph - 1u : 0xffffffffu;
    return g;
}
__host__ __device__ inline uint32_t phys_col(const MapGeom& g, uint32_t x) { return x & g.xmask; }
// Band extents. Besides its bounding box, every slot records per band of 8 rows the column range
// [x0, x1) (multiples of 8) that may hold informed cells, packed x0 | x1 << 16, 0 = nothing in this
// band. Walls occlude most of a lidar's disc: summed over the bands the ranges cover ~58 % of the
// box, and that is all the resampler moves. Entries are indexed by the PHYSICAL band of the slot
// and are 0 for every band outside the box's rows (invariant kept by init, ray update and copy).
constexpr int BAND_ROWS = 8;
__host__ __device__ inline uint32_t bands_per_slot(const MapGeom& g) { return (g.ph + BAND_ROWS - 1u) / BAND_ROWS; }
__host__ __device__ inline uint32_t phys_band(const MapGeom& g, uint32_t y) { return (y & g.ymask) / BAND_ROWS; }
// offset of logical cell (x, y) inside a slot
__host__ __device__ inline size_t phys_index(const MapGeom& g, uint32_t x, uint32_t y) {
    const uint32_t py = y & g.ymask, px = phys_col(g, x);
    if (g.tiled)
        return ((size_t)(py / TILE_ROWS) * g.tiles_per_row + px / TILE_COLS) * TILE_CELLS + (py % TILE_ROWS) * TILE_COLS +
               px % TILE_COLS;
    return (size_t)py * g.pw + px;
}

// offset, in 32-byte units (8 cells), of unit `u` of slot row `py`
__host__ __device__ inline uint32_t phys_unit(const MapGeom& g, uint32_t py, uint32_t u) {
    if (g.tiled)
        return ((py / TILE_ROWS) * g.tiles_per_row + u / (TILE_COLS / 8u)) * (TILE_CELLS / 8u) +
               (py % TILE_ROWS) * (TILE_COLS / 8u) + u % (TILE_COLS / 8u);
    return py * (g.pw / 8u) + u;
}

// Map::world_to_grid, map.rs:60-62
__device__ __forceinline__ float world_to_grid(float w, float pos, float res) {
    return __fdiv_rn(__fsub_rn(w, pos), res);
}
// Map::is_valid, map.rs:64-69
__device__ __forceinline__ bool grid_is_valid(float gx, float gy, uint32_t gw, uint32_t gh) {
    return !((gx < 0.0f) || (gy < 0.0f) || (f32_as_usize(gx) >= (unsigned long long)gw) ||
             (f32_as_usize(gy) >= (unsigned long long)gh));
}

// beam endpoint in world coordinates, map.rs:75-78 / 120-123
__device__ __forceinline__ void beam_endpoint(float px, float py, float ptheta, float angle, float dist, float* ex,
                                              float* ey) {
    const float a = __fadd_rn(ptheta, angle);
    float sn, cs;
    slamrs_libm::sincosf_exact(a, &sn, &cs);
    *ex = __fadd_rn(px, __fmul_rn(cs, dist));
    *ey = __fadd_rn(py, __fmul_rn(sn, dist));
}

// inverse_sensor_model, map.rs:148-172 with tolerance 2.0 (map.rs:104).
// returns the packed counter increment: 0 (prior), CELL_FREE_INC or CELL_OCC_INC
__device__ __forceinline__ uint32_t inverse_sensor_increment(float distance, float measured, bool was_hit) {
    if (!was_hit) return (distance < measured) ? CELL_FREE_INC : 0u;
    const float half_tol = __fdiv_rn(2.0f, 2.0f);
    if (distance < __fsub_rn(measured, half_tol)) return CELL_FREE_INC;
    if (distance > __fadd_rn(measured, half_tol)) return 0u;
    return CELL_OCC_INC;
}

// ---------------------------------------------------------------------------- ray iterator
// GridRayIterator::new + next, slamrs/slam/src/grid/ray.rs:21-77, 83-110, fused with the
// squared start-to-cell-centre distance that apply_measurement needs (map.rs:99-100).
// `visit(x, y, acc)` is called for every emitted cell, in order, where
//     acc = fl(fl(dx*dx) + fl(dy*dy)),  dx = fl(x0 - (x + 0.5)),  dy = fl(y0 - (y + 0.5))
// is exactly the value nalgebra's EuclideanNorm folds before taking the square root
// (0 + dx^2 is exact). The running `error` term is a sequential f32 accumulation and is not
// re-associated. Cell centres x + 0.5 are exact in f32 for |x| < 2^22, so they are carried
// incrementally (+-1 per step, exact) and only the coordinate that moved is recomputed.
template <typename Visit>
__device__ __forceinline__ void ray_walk_acc(float x0, float y0, float x1, float y1, uint32_t size_x, uint32_t size_y,
                                             uint32_t additional_steps, Visit&& visit) {
    const float delta_x = fabsf(__fsub_rn(x1, x0));
    const float delta_y = fabsf(__fsub_rn(y1, y0));
    const float fx0 = floorf(x0), fy0 = floorf(y0);
    const long long sx = f32_as_isize(fx0);
    const long long sy = f32_as_isize(fy0);
    // A start outside the grid emits nothing (ray.rs:88-92 fails on the first call).
    if (sx < 0 || sx >= (long long)size_x || sy < 0 || sy >= (long long)size_y) return;

    unsigned long long n = 1ull + additional_steps;  // wrapping isize arithmetic, then `as usize`
    int x_inc, y_inc;
    float error;
    if (delta_x == 0.0f) {
        x_inc = 0;
        error = __int_as_float(0x7f800000);
    } else if (x1 > x0) {
        x_inc = 1;
        n += (unsigned long long)f32_as_isize(__fsub_rn(floorf(x1), (float)sx));
        error = __fmul_rn(__fsub_rn(__fadd_rn(fx0, 1.0f), x0), delta_y);
    } else {
        x_inc = -1;
        n += (unsigned long long)sx - (unsigned long long)f32_as_isize(floorf(x1));
        error = __fmul_rn(__fsub_rn(x0, fx0), delta_y);
    }
    if (delta_y == 0.0f) {
        y_inc = 0;
        error = __fsub_rn(error, __int_as_float(0x7f800000));
    } else if (y1 > y0) {
        y_inc = 1;
        n += (unsigned long long)f32_as_isize(floorf(y1)) - (unsigned long long)sy;
        error = __fsub_rn(error, __fmul_rn(__fsub_rn(__fadd_rn(fy0, 1.0f), y0), delta_x));
    } else {
        y_inc = -1;
        n += (unsigned long long)sy - (unsigned long long)f32_as_isize(floorf(y1));
        error = __fsub_rn(error, __fmul_rn(__fsub_rn(y0, fy0), delta_x));
    }
    // The walk stops at the first cell outside the grid, and a step that cannot move
    // (increment 0 on the chosen axis) only happens with n <= 3 + size_y, so
    // size_x + size_y + 8 bounds the trip count without changing the emitted sequence.
    const unsigned long long cap = (unsigned long long)size_x + size_y + 8ull;
    int remaining = (int)(n < cap ? n : cap);
    int x = (int)sx, y = (int)sy;
    const float x_step = (float)x_inc, y_step = (float)y_inc;
    float cx = __fadd_rn((float)x, 0.5f), cy = __fadd_rn((float)y, 0.5f);
    float dx = __fsub_rn(x0, cx), dy = __fsub_rn(y0, cy);
    float dx2 = __fmul_rn(dx, dx), dy2 = __fmul_rn(dy, dy);
    bool inside = true;
    while (remaining > 0 && inside) {
        visit(x, y, __fadd_rn(dx2, dy2));
        if (error > 0.0f) {
            y += y_inc;
            error = __fsub_rn(error, delta_x);
            cy = __fadd_rn(cy, y_step);
            dy = __fsub_rn(y0, cy);
            dy2 = __fmul_rn(dy, dy);
            inside = (unsigned)y < size_y;
        } else {
            x += x_inc;
            error = __fadd_rn(error, delta_y);
            cx = __fadd_rn(cx, x_step);
            dx = __fsub_rn(x0, cx);
            dx2 = __fmul_rn(dx, dx);
            inside = (unsigned)x < size_x;
        }
        remaining -= 1;
    }
}

template <typename Visit>
__device__ __forceinline__ void ray_walk(float x0, float y0, float x1, float y1, uint32_t size_x, uint32_t size_y,
                                         uint32_t additional_steps, Visit&& visit) {
    ray_walk_acc(x0, y0, x1, y1, size_x, size_y, additional_steps, [&](int x, int y, float) { visit(x, y); });
}

// ---- inverse sensor model without the per-cell square root ---------------------------------
// inverse_sensor_model (map.rs:148-172) compares distance = fl(sqrt(acc)) with thresholds that
// are constant along a ray. IEEE sqrt is correctly rounded and monotone, so each comparison
// can be moved into the acc domain once per ray:
//     fl(sqrt(a)) <  t   <=>   a <  acc_threshold_below(t)
//     fl(sqrt(a)) >  t   <=>   a >  acc_threshold_above(t)
// for every a >= 0 (including +inf); NaN a or NaN t make both sides false, as in the reference.
__device__ __forceinline__ float f32_next_up(float a) {    // a >= 0, finite or inf
    return a == __int_as_float(0x7f800000) ? a : __int_as_float(__float_as_int(a) + 1);
}
__device__ __forceinline__ float f32_next_down(float a) {  // a > 0
    return __int_as_float(__float_as_int(a) - 1);
}
// smallest A >= 0 with fl(sqrt(A)) >= t  (so that d < t  <=>  acc < A)
__device__ __forceinline__ float acc_threshold_below(float t) {
    if (!(t > 0.0f)) return 0.0f;                       // t <= 0 or NaN: d < t never holds
    if (t == __int_as_float(0x7f800000)) return t;      // d < inf  <=>  acc < inf
    float a = __fmul_rn(t, t);                          // may be +inf or underflow to 0
    while (a > 0.0f && __fsqrt_rn(f32_next_down(a)) >= t) a = f32_next_down(a);
    while (__fsqrt_rn(a) < t) a = f32_next_up(a);       // sqrt(+inf) = +inf >= t terminates
    return a;
}
// largest B with fl(sqrt(B)) <= t  (so that d > t  <=>  acc > B); -1 when every acc >= 0 exceeds it
__device__ __forceinline__ float acc_threshold_above(float t) {
    if (t != t) return __int_as_float(0x7f800000);      // NaN: d > t never holds
    if (t < 0.0f) return -1.0f;                         // d >= 0 > t always
    if (t == __int_as_float(0x7f800000)) return t;      // d > inf never
    float b = __fmul_rn(t, t);
    if (b == __int_as_float(0x7f800000)) b = __int_as_float(0x7f7fffff);
    while (__fsqrt_rn(b) > t) b = f32_next_down(b);     // t >= 0: sqrt(0) = 0 <= t terminates
    while (b < __int_as_float(0x7f7fffff) && __fsqrt_rn(f32_next_up(b)) <= t) b = f32_next_up(b);
    return b;
}

struct RayClassifier {   // per-ray constants of inverse_sensor_model with tolerance 2.0 (map.rs:104)
    float free_below;    // acc <  free_below -> P_FREE
    float prior_above;   // acc >  prior_above -> P_PRIOR
    uint32_t mid_inc;    // otherwise: P_OCCUPPIED for a hit, P_PRIOR for a miss
};
__device__ __forceinline__ RayClassifier make_ray_classifier(float measured, bool was_hit) {
    RayClassifier c;
    if (!was_hit) {  // free strictly before the reading, prior from there on
        c.free_below = acc_threshold_below(measured);
        c.prior_above = __int_as_float(0x7f800000);
        c.mid_inc = 0u;
    } else {
        const float half_tol = __fdiv_rn(2.0f, 2.0f);
        c.free_below = acc_threshold_below(__fsub_rn(measured, half_tol));
        c.prior_above = acc_threshold_above(__fadd_rn(measured, half_tol));
        c.mid_inc = CELL_OCC_INC;
    }
    return c;
}
__device__ __forceinline__ uint32_t classify_cell(const RayClassifier& c, float acc) {
    if (acc < c.free_below) return CELL_FREE_INC;
    if (acc > c.prior_above) return 0u;
    return c.mid_inc;
}

// ---------------------------------------------------------------------------- motion model
struct OdomModel {  // Odometry::new, robot.rs:132-150
    double mean_c, std_c, mean_t, std_t;
};

// statrs 0.18 Normal::pdf: exp(-0.5 d d) / (sqrt(2 pi) sigma), d = (x - mean) / sigma
__device__ __forceinline__ double normal_pdf(double x, double mean, double sd) {
    const double SQRT_2PI = 2.5066282746310005024157652848110452530069867406099;
    const double d = __ddiv_rn(__dsub_rn(x, mean), sd);
    return __ddiv_rn(exp(__dmul_rn(__dmul_rn(-0.5, d), d)), __dmul_rn(SQRT_2PI, sd));
}

// angle_diff, common/src/math.rs:150-157 (Rust % on f64 == fmod)
__device__ __forceinline__ double angle_diff(double alpha, double beta) {
    const double PI = 3.14159265358979323846264338327950288;
    const double diff = __dsub_rn(fmod(__dadd_rn(__dsub_rn(beta, alpha), PI), __dmul_rn(PI, 2.0)), PI);
    if (diff < -PI) return __dadd_rn(diff, __dmul_rn(2.0, PI));
    return diff;
}

// f64::total_cmp key: monotone map from the IEEE bit pattern to a signed integer
__device__ __forceinline__ long long total_order_key(double v) {
    long long b = __double_as_longlong(v);
    b ^= (long long)(((unsigned long long)(b >> 63)) >> 1);
    return b;
}

}  // namespace slamrs
