/* ============================================================================================
 * TEST INFRASTRUCTURE ONLY -- CPU oracle of the localiser: GridMapSlam::update (slam.rs:46-75) with
 * one fixed map shared by every particle, externalised draws and the optional adaptive resampling
 * of slam_oracle.c. Motion (so_odometry_sample / so_odometry_log_prob) and the fold
 * (so_resample_fold) are slam_oracle.c's; the beam term is read from a per-cell table:
 *   beam endpoint     (p == 0.5) ? 0 : log(0.9 p + 0.1), 0 off the grid      (map.rs:130-141)
 *   likelihood field  log(z_hit exp(((-0.5 d2) res^2) / sigma^2) + z_rand), log(z_rand) off the grid,
 *                     d2 = exact squared distance in cells to the nearest cell with p > occupied_above
 * The distance is found by an exhaustive search, independent of the device's two-pass transform.
 * Build flags as slam_oracle.c: no contraction, no fast math.
 * ============================================================================================ */
#include "loc_oracle.h"

#include <math.h>
#include <stdlib.h>
#include <string.h>

struct so_loc {
    uint64_t n, gw, gh;
    float pos_x, pos_y, res;
    double* terms;
    double outside;
    so_pose* pose;
    double* weight;
    double* raw_weight;
    double* own_raw;
    uint64_t* last_idx;
    uint64_t max_particle;
    double adaptive_tau;
    double* carry;
    int resampled;
    const double* weight_override;
};

/* f32 as usize, saturating, NaN -> 0 */
static inline uint64_t as_usize(float v) {
    if (!(v == v) || v <= 0.0f) return 0;
    if (v >= 18446744073709551616.0f) return UINT64_MAX;
    return (uint64_t)v;
}

/* For every cell, every obstacle row is visited outward from the cell's row (the row distance alone bounds the
 * rest); in each row the nearest obstacle column comes from a bisection of that row's sorted obstacle columns. */
int64_t so_loc_distance2(const double* map, uint64_t gw, uint64_t gh, double occupied_above, int64_t* out) {
    const uint64_t cells = gw * gh;
    uint64_t* start = (uint64_t*)calloc(gh + 1, sizeof(uint64_t));
    int64_t* cols = (int64_t*)malloc((cells ? cells : 1) * sizeof(int64_t));
    if (!start || !cols) abort();
    int64_t n_obst = 0;
    for (uint64_t row = 0; row < gh; ++row) {
        start[row] = (uint64_t)n_obst;
        for (uint64_t col = 0; col < gw; ++col)
            if (map[row * gh + col] > occupied_above) cols[n_obst++] = (int64_t)col;   /* ascending */
    }
    start[gh] = (uint64_t)n_obst;
    for (uint64_t row = 0; row < gh; ++row) {
        for (uint64_t col = 0; col < gw; ++col) {
            int64_t best = -1;
            for (uint64_t k = 0; k < gh; ++k) {
                const int64_t k2 = (int64_t)(k * k);
                if (best >= 0 && k2 >= best) break;
                for (int side = 0; side < 2; ++side) {
                    if (side == 1 && k == 0) break;
                    const int64_t r = side ? (int64_t)row + (int64_t)k : (int64_t)row - (int64_t)k;
                    if (r < 0 || r >= (int64_t)gh) continue;
                    uint64_t lo = start[r], hi = start[r + 1];
                    if (lo == hi) continue;
                    while (lo < hi) {   /* first obstacle column >= col */
                        const uint64_t mid = lo + (hi - lo) / 2;
                        if (cols[mid] < (int64_t)col) lo = mid + 1; else hi = mid;
                    }
                    for (uint64_t c = (lo > start[r] ? lo - 1 : lo); c <= lo && c < start[r + 1]; ++c) {
                        const int64_t dx = cols[c] - (int64_t)col;
                        const int64_t d2 = dx * dx + k2;
                        if (best < 0 || d2 < best) best = d2;
                    }
                }
            }
            out[row * gh + col] = best;
        }
    }
    free(start);
    free(cols);
    return n_obst;
}

struct so_loc* so_loc_create(float pos_x, float pos_y, float resolution, uint64_t gw, uint64_t gh, uint64_t n_particles,
                             int kind, float sigma, float z_rand, float occupied_above, const double* map) {
    if (n_particles == 0 || gw == 0 || gw != gh) return NULL;
    struct so_loc* s = (struct so_loc*)calloc(1, sizeof(*s));
    if (!s) return NULL;
    s->n = n_particles; s->gw = gw; s->gh = gh;
    s->pos_x = pos_x; s->pos_y = pos_y; s->res = resolution;
    const uint64_t cells = gw * gh;
    s->terms = (double*)malloc(cells * sizeof(double));
    s->pose = (so_pose*)calloc(n_particles, sizeof(so_pose));
    s->weight = (double*)malloc(n_particles * sizeof(double));
    s->raw_weight = (double*)malloc(n_particles * sizeof(double));
    s->own_raw = (double*)calloc(n_particles, sizeof(double));
    s->last_idx = (uint64_t*)calloc(n_particles, sizeof(uint64_t));
    if (!s->terms || !s->pose || !s->weight || !s->raw_weight || !s->own_raw || !s->last_idx) { so_loc_destroy(s); return NULL; }
    for (uint64_t i = 0; i < n_particles; ++i) { s->weight[i] = s->raw_weight[i] = 1.0 / (double)n_particles; s->last_idx[i] = i; }
    if (kind == 0) {
        const double Z_HIT = 0.9, SENSOR_MAXDIST = 1.0;
        for (uint64_t c = 0; c < cells; ++c)
            s->terms[c] = map[c] == 0.5 ? log(1.0 / SENSOR_MAXDIST) : log(Z_HIT * map[c] + (1.0 - Z_HIT) * 1.0 / SENSOR_MAXDIST);
        s->outside = 0.0;
    } else {
        const double zr = (double)z_rand, zh = 1.0 - zr, rr = (double)resolution * (double)resolution;
        const double ss = (double)sigma * (double)sigma;
        int64_t* d2 = (int64_t*)malloc(cells * sizeof(int64_t));
        if (!d2) { so_loc_destroy(s); return NULL; }
        so_loc_distance2(map, gw, gh, (double)occupied_above, d2);
        for (uint64_t c = 0; c < cells; ++c)
            s->terms[c] = d2[c] < 0 ? log(zr) : log(zh * exp(((-0.5 * (double)d2[c]) * rr) / ss) + zr);
        free(d2);
        s->outside = log(zr);
    }
    return s;
}

void so_loc_destroy(struct so_loc* s) {
    if (!s) return;
    free(s->terms); free(s->pose); free(s->weight); free(s->raw_weight); free(s->own_raw); free(s->last_idx); free(s->carry);
    free(s);
}

void so_loc_terms(const struct so_loc* s, double* out) { memcpy(out, s->terms, s->gw * s->gh * sizeof(double)); }
double so_loc_outside(const struct so_loc* s) { return s->outside; }
void so_loc_set_adaptive_resampling(struct so_loc* s, double tau) { s->adaptive_tau = tau; }
int so_loc_resampled(const struct so_loc* s) { return s->resampled; }
/* resample the next update on these raw weights (the device's), as so_set_weight_override does for the SLAM oracle */
void so_loc_set_weight_override(struct so_loc* s, const double* raw) { s->weight_override = raw; }
void so_loc_get_own_raw(const struct so_loc* s, double* out) { memcpy(out, s->own_raw, s->n * sizeof(double)); }

int so_loc_update(struct so_loc* s, const double* angle, const double* dist, const uint8_t* valid, uint64_t nb, float dl,
                  float dr, float wheel, const double* z, double u01) {
    double od[4];
    so_odometry_new(dl, dr, wheel, od);
    const uint64_t n = s->n;
    for (uint64_t p = 0; p < n; ++p) {
        const so_pose initial = s->pose[p];
        const so_pose np = so_odometry_sample(od, initial, z[2 * p], z[2 * p + 1]);
        double lp = log(1.0);
        for (uint64_t i = 0; i < nb; ++i) {
            if (!valid[i]) continue;
            const float a = np.theta + (float)angle[i];
            const float ex = np.x + cosf(a) * (float)dist[i];
            const float ey = np.y + sinf(a) * (float)dist[i];
            const float gx = (ex - s->pos_x) / s->res, gy = (ey - s->pos_y) / s->res;
            const int inside = !((gx < 0.0f) || (gy < 0.0f) || (as_usize(gx) >= s->gw) || (as_usize(gy) >= s->gh));
            lp += inside ? s->terms[as_usize(gy) * s->gh + as_usize(gx)] : s->outside;
        }
        s->raw_weight[p] = exp(lp + so_odometry_log_prob(od, initial, np));
        s->pose[p] = np;
    }
    if (s->carry)
        for (uint64_t p = 0; p < n; ++p) s->raw_weight[p] = s->carry[p] * s->raw_weight[p];
    memcpy(s->own_raw, s->raw_weight, n * sizeof(double));
    if (s->weight_override) {
        memcpy(s->raw_weight, s->weight_override, n * sizeof(double));
        s->weight_override = NULL;
    }
    const int clamped = so_resample_fold(s->raw_weight, n, u01, s->weight, NULL, s->last_idx, &s->max_particle);
    s->resampled = 1;
    if (s->adaptive_tau > 0.0) {
        double sq = 0.0;
        for (uint64_t p = 0; p < n; ++p) sq += s->weight[p] * s->weight[p];
        if (!(1.0 / sq < s->adaptive_tau * (double)n)) {
            if (!s->carry) s->carry = (double*)malloc(n * sizeof(double));
            memcpy(s->carry, s->weight, n * sizeof(double));
            for (uint64_t p = 0; p < n; ++p) s->last_idx[p] = p;
            s->resampled = 0;
            return 0;
        }
        free(s->carry);
        s->carry = NULL;
    }
    so_pose* next = (so_pose*)malloc(n * sizeof(so_pose));
    if (!next) return -1;
    for (uint64_t m = 0; m < n; ++m) next[m] = s->pose[s->last_idx[m]];
    free(s->pose);
    s->pose = next;
    return clamped;
}

void so_loc_get_poses(const struct so_loc* s, float* out) {
    for (uint64_t i = 0; i < s->n; ++i) { out[3 * i] = s->pose[i].x; out[3 * i + 1] = s->pose[i].y; out[3 * i + 2] = s->pose[i].theta; }
}
void so_loc_set_poses(struct so_loc* s, const float* xyt) {
    for (uint64_t i = 0; i < s->n; ++i) { s->pose[i].x = xyt[3 * i]; s->pose[i].y = xyt[3 * i + 1]; s->pose[i].theta = xyt[3 * i + 2]; }
}
void so_loc_get_weights(const struct so_loc* s, double* norm, double* raw) {
    if (norm) memcpy(norm, s->weight, s->n * sizeof(double));
    if (raw) memcpy(raw, s->raw_weight, s->n * sizeof(double));
}
void so_loc_get_indices(const struct so_loc* s, uint64_t* idx) { memcpy(idx, s->last_idx, s->n * sizeof(uint64_t)); }
uint64_t so_loc_max_particle(const struct so_loc* s) { return s->max_particle; }
/* estimated_pose, slam.rs:77-81: the new generation indexed by the pre-resample argmax */
so_pose so_loc_estimated_pose(const struct so_loc* s) { return s->pose[s->max_particle]; }
double so_loc_effective_particles(const struct so_loc* s) {
    double sum = 0.0;
    for (uint64_t i = 0; i < s->n; ++i) sum += s->weight[i] * s->weight[i];
    return 1.0 / sum;
}
