/* ============================================================================================
 * TEST INFRASTRUCTURE ONLY -- CPU oracle of the localiser's KLD-sampling (adaptive population,
 * slamrs_gpu_set_kld): a variable-population restatement of the localiser update. Motion is
 * slam_oracle.c's (so_odometry_sample / so_odometry_log_prob), the per-cell term table is
 * loc_oracle.c's (so_loc_terms / so_loc_outside), recovery is recovery_oracle.c's
 * (so_recovery_update / ss_recovery_draw). Added here: the bin of a pose, AMCL's bound on the
 * number of particles and the fold that draws M particles from N weights. Build flags as
 * slam_oracle.c: no contraction, no fast math.
 * ============================================================================================ */
#include "kld_oracle.h"

#include <math.h>
#include <stdlib.h>
#include <string.h>

#include "loc_oracle.h"
#include "recovery_oracle.h"

static const double TWO_PI = 0x1.921fb54442d18p+2;

/* f32 as usize, saturating, NaN -> 0 */
static inline uint64_t as_usize(float v) {
    if (!(v == v) || v <= 0.0f) return 0;
    if (v >= 18446744073709551616.0f) return UINT64_MAX;
    return (uint64_t)v;
}

/* f64::total_cmp */
static inline int total_cmp(double a, double b) {
    int64_t x, y;
    memcpy(&x, &a, 8); memcpy(&y, &b, 8);
    x ^= (int64_t)((uint64_t)(x >> 63) >> 1);
    y ^= (int64_t)((uint64_t)(y >> 63) >> 1);
    return (x > y) - (x < y);
}

uint64_t so_kld_bin(float x, float y, float theta, float pos_x, float pos_y, float res, uint64_t gw, uint64_t gh,
                    uint32_t bin_cells, uint32_t theta_bins) {
    const uint64_t nbx = (gw + bin_cells - 1) / bin_cells, nby = (gh + bin_cells - 1) / bin_cells;
    const float gx = (x - pos_x) / res, gy = (y - pos_y) / res;
    if ((gx < 0.0f) || (gy < 0.0f) || as_usize(gx) >= gw || as_usize(gy) >= gh) return nbx * nby * theta_bins;
    double t = fmod((double)theta, TWO_PI);
    if (t < 0.0) t += TWO_PI;
    uint64_t h = 0;
    if (t >= 0.0 && t < TWO_PI) {
        h = (uint64_t)((t * (double)theta_bins) / TWO_PI);
        if (h > theta_bins - 1u) h = theta_bins - 1u;
    }
    return ((as_usize(gy) / bin_cells) * nbx + as_usize(gx) / bin_cells) * theta_bins + h;
}

uint64_t so_kld_count(const float* xyt, uint64_t n, float pos_x, float pos_y, float res, uint64_t gw, uint64_t gh,
                      uint32_t bin_cells, uint32_t theta_bins) {
    const uint64_t nb = (gw + bin_cells - 1) / bin_cells;
    const uint64_t bins = nb * ((gh + bin_cells - 1) / bin_cells) * theta_bins + 1;
    uint8_t* seen = (uint8_t*)calloc((size_t)((bins + 7) / 8), 1);
    if (!seen) abort();
    uint64_t k = 0;
    for (uint64_t i = 0; i < n; ++i) {
        const uint64_t b = so_kld_bin(xyt[3 * i], xyt[3 * i + 1], xyt[3 * i + 2], pos_x, pos_y, res, gw, gh, bin_cells,
                                      theta_bins);
        if (!(seen[b >> 3] & (1u << (b & 7)))) { seen[b >> 3] |= (uint8_t)(1u << (b & 7)); ++k; }
    }
    free(seen);
    return k;
}

/* pf_resample_limit (AMCL pf.c) in its order of operations */
uint64_t so_kld_bound(uint64_t k, uint64_t n_min, uint64_t n_max, double err, double z) {
    if (k <= 1) return n_min;
    const double km1 = (double)(k - 1);
    const double b = 2.0 / (9.0 * km1);
    const double x = 1.0 - b + sqrt(b) * z;
    const double n = (km1 / (2.0 * err)) * x * x * x;
    if (!(n < (double)n_max)) return n_max;
    const double c = ceil(n);
    return c < (double)n_min ? n_min : (uint64_t)c;
}

int so_resample_fold_m(const double* raw, uint64_t n, uint64_t m, double u01, double* norm, uint64_t* idx,
                       uint64_t* max_particle) {
    /* normalize_weights, particle.rs:49-56 */
    double sum = 0.0;
    for (uint64_t p = 0; p < n; ++p) sum += raw[p];
    for (uint64_t p = 0; p < n; ++p) norm[p] = raw[p] / sum;
    /* max_by(total_cmp): last maximum wins, particle.rs:40-46 */
    uint64_t best = 0;
    for (uint64_t p = 1; p < n; ++p)
        if (total_cmp(norm[p], norm[best]) >= 0) best = p;
    *max_particle = best;
    /* resample, particle.rs:78-101, with m wherever N counts draws */
    int clamped = 0;
    const double num = (double)m;
    const double r = u01 * 1.0 / num;
    double c = norm[0];
    uint64_t i = 0;
    for (uint64_t mm = 1; mm <= m; ++mm) {
        const double u = r + ((double)mm - 1.0) * 1.0 / num;
        while (u > c) {
            if (i + 1 >= n) { clamped = 1; break; }
            i += 1;
            c += norm[i];
        }
        idx[mm - 1] = i;
    }
    return clamped;
}

struct so_kld {
    uint64_t cap, n, gw, gh;
    float pos_x, pos_y, res;
    double* terms;
    double outside;
    so_pose* pose;          /* the current generation: n of cap */
    so_pose* next;          /* scratch */
    double *norm, *raw, *own_raw;
    uint64_t* idx;
    uint64_t max_particle, n_weighted, k, m_drawn;
    so_pose est;
    int has_est;
    int kld_on, kld_last;
    uint64_t n_min, n_max;
    double err, z;
    uint32_t bin_cells, theta_bins;
    int rec_on, rec_last;
    double alpha_slow, alpha_fast, w_slow, w_fast, p;
    uint64_t seed, injected;
    uint32_t* free_cells;
    uint32_t n_free;
    uint64_t step;
    const double* weight_override;
};

struct so_kld* so_kld_create(float pos_x, float pos_y, float resolution, uint64_t gw, uint64_t gh, uint64_t n_particles,
                             int kind, float sigma, float z_rand, float occupied_above, const double* map) {
    if (n_particles == 0 || gw == 0 || gw != gh) return NULL;
    struct so_kld* s = (struct so_kld*)calloc(1, sizeof(*s));
    if (!s) return NULL;
    const uint64_t cells = gw * gh, n = n_particles;
    s->cap = s->n = s->n_weighted = s->m_drawn = n;
    s->gw = gw; s->gh = gh;
    s->pos_x = pos_x; s->pos_y = pos_y; s->res = resolution;
    s->terms = (double*)malloc(cells * sizeof(double));
    s->pose = (so_pose*)calloc(n, sizeof(so_pose));
    s->next = (so_pose*)calloc(n, sizeof(so_pose));
    s->norm = (double*)malloc(n * sizeof(double));
    s->raw = (double*)malloc(n * sizeof(double));
    s->own_raw = (double*)calloc(n, sizeof(double));
    s->idx = (uint64_t*)calloc(n, sizeof(uint64_t));
    s->free_cells = (uint32_t*)malloc(cells * sizeof(uint32_t));
    /* the term table of the localiser oracle (one particle: only its table is used) */
    struct so_loc* loc = so_loc_create(pos_x, pos_y, resolution, gw, gh, 1, kind, sigma, z_rand, occupied_above, map);
    if (!s->terms || !s->pose || !s->next || !s->norm || !s->raw || !s->own_raw || !s->idx || !s->free_cells || !loc) {
        so_loc_destroy(loc);
        so_kld_destroy(s);
        return NULL;
    }
    so_loc_terms(loc, s->terms);
    s->outside = so_loc_outside(loc);
    so_loc_destroy(loc);
    for (uint64_t i = 0; i < n; ++i) { s->norm[i] = s->raw[i] = 1.0 / (double)n; s->idx[i] = i; }
    for (uint64_t c = 0; c < cells; ++c)
        if (map[c] < 0.5) s->free_cells[s->n_free++] = (uint32_t)c;
    return s;
}

void so_kld_destroy(struct so_kld* s) {
    if (!s) return;
    free(s->terms); free(s->pose); free(s->next); free(s->norm); free(s->raw); free(s->own_raw); free(s->idx);
    free(s->free_cells);
    free(s);
}

void so_kld_set_kld(struct so_kld* s, int on, uint64_t n_min, uint64_t n_max, double err, double z, uint32_t bin_cells,
                    uint32_t theta_bins) {
    s->kld_on = on;
    s->n_min = n_min; s->n_max = n_max; s->err = err; s->z = z; s->bin_cells = bin_cells; s->theta_bins = theta_bins;
}

void so_kld_set_recovery(struct so_kld* s, double alpha_slow, double alpha_fast, uint64_t seed) {
    s->rec_on = alpha_fast > 0.0;
    s->alpha_slow = alpha_slow; s->alpha_fast = alpha_fast; s->seed = seed;
    s->w_slow = s->w_fast = s->p = 0.0;
    s->injected = 0;
    s->rec_last = 0;
}

void so_kld_set_weight_override(struct so_kld* s, const double* raw) { s->weight_override = raw; }

int so_kld_update(struct so_kld* s, const double* angle, const double* dist, const uint8_t* valid, uint64_t nb, float dl,
                  float dr, float wheel, const double* z, double u01) {
    const uint64_t step = s->step++;
    const uint64_t n = s->n;
    uint64_t m = s->cap, k = 0;
    if (s->kld_on) {   /* the bins of the generation this update starts from */
        float* xyt = (float*)malloc(n * 3 * sizeof(float));
        if (!xyt) return -1;
        so_kld_get_poses(s, xyt);
        k = so_kld_count(xyt, n, s->pos_x, s->pos_y, s->res, s->gw, s->gh, s->bin_cells, s->theta_bins);
        free(xyt);
        m = so_kld_bound(k, s->n_min, s->n_max, s->err, s->z);
    }
    /* motion and likelihood, loc_oracle.c's so_loc_update over the n particles */
    double od[4];
    so_odometry_new(dl, dr, wheel, od);
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
        s->raw[p] = exp(lp + so_odometry_log_prob(od, initial, np));
        s->pose[p] = np;
    }
    memcpy(s->own_raw, s->raw, n * sizeof(double));
    if (s->weight_override) {
        memcpy(s->raw, s->weight_override, n * sizeof(double));
        s->weight_override = NULL;
    }
    const int clamped = so_resample_fold_m(s->raw, n, m, u01, s->norm, s->idx, &s->max_particle);
    for (uint64_t j = 0; j < m; ++j) s->next[j] = s->pose[s->idx[j]];
    so_pose* t = s->pose; s->pose = s->next; s->next = t;
    /* estimated_pose: the reference's new[max_particle] at the same cumulative-mass position of m draws */
    s->est = s->pose[s->max_particle * m / n];
    s->has_est = 1;
    s->n = m; s->n_weighted = n; s->m_drawn = m; s->k = k;
    s->kld_last = s->kld_on;
    /* recovery (recovery_oracle.c's so_rec_update): the averages over the n weighted, injection over the m drawn */
    s->p = 0.0;
    s->injected = 0;
    s->rec_last = s->rec_on;
    if (!s->rec_on) return clamped;
    double sum = 0.0;
    for (uint64_t i = 0; i < n; ++i) sum += s->raw[i];
    s->p = so_recovery_update(sum, n, s->alpha_slow, s->alpha_fast, &s->w_slow, &s->w_fast);
    if (!(s->p > 0.0)) return clamped;
    for (uint64_t j = 0; j < m; ++j) {
        float q[3];
        if (ss_recovery_draw(s->seed, step, j, s->p, s->free_cells, s->n_free, s->gh, (double)s->pos_x, (double)s->pos_y,
                             (double)s->res, q)) {
            s->pose[j].x = q[0]; s->pose[j].y = q[1]; s->pose[j].theta = q[2];
            ++s->injected;
        }
    }
    return clamped;
}

uint64_t so_kld_population(const struct so_kld* s) { return s->n; }

void so_kld_state(const struct so_kld* s, uint64_t* out3) {
    out3[0] = s->kld_last ? s->n_weighted : 0;
    out3[1] = s->kld_last ? s->k : 0;
    out3[2] = s->kld_last ? s->m_drawn : 0;
}

void so_kld_recovery_state(const struct so_kld* s, double* out3, uint64_t* injected) {
    out3[0] = s->rec_last ? s->w_slow : 0.0;
    out3[1] = s->rec_last ? s->w_fast : 0.0;
    out3[2] = s->rec_last ? s->p : 0.0;
    if (injected) *injected = s->rec_last ? s->injected : 0;
}

void so_kld_get_poses(const struct so_kld* s, float* out) {
    for (uint64_t i = 0; i < s->n; ++i) { out[3 * i] = s->pose[i].x; out[3 * i + 1] = s->pose[i].y; out[3 * i + 2] = s->pose[i].theta; }
}
void so_kld_set_poses(struct so_kld* s, const float* xyt) {
    for (uint64_t i = 0; i < s->n; ++i) { s->pose[i].x = xyt[3 * i]; s->pose[i].y = xyt[3 * i + 1]; s->pose[i].theta = xyt[3 * i + 2]; }
}
void so_kld_get_weights(const struct so_kld* s, double* norm, double* raw) {
    if (norm) memcpy(norm, s->norm, s->n_weighted * sizeof(double));
    if (raw) memcpy(raw, s->raw, s->n_weighted * sizeof(double));
}
void so_kld_get_own_raw(const struct so_kld* s, double* out) { memcpy(out, s->own_raw, s->n_weighted * sizeof(double)); }
void so_kld_get_indices(const struct so_kld* s, uint64_t* idx) { memcpy(idx, s->idx, s->m_drawn * sizeof(uint64_t)); }
uint64_t so_kld_max_particle(const struct so_kld* s) { return s->max_particle; }
so_pose so_kld_estimated_pose(const struct so_kld* s) { return s->has_est ? s->est : s->pose[s->max_particle]; }
