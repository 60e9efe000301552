/* ============================================================================================
 * TEST INFRASTRUCTURE ONLY -- CPU oracle of the localiser's recovery (augmented MCL,
 * slamrs_gpu_set_recovery). It wraps the localiser oracle of loc_oracle.c: after each of its updates
 * (motion, likelihood, resampling) it records the estimate, updates the averages of the raw weights
 * from their left fold and replaces new particles by poses in the map's free cells, drawn from the
 * shared stream (counter domains 4, 5 and 6). Restates slamrs_stream::recovery_update / recovery_slot /
 * recovery_draw of slamrs_b200/csrc/shared_stream.cuh. Build flags as slam_oracle.c: no contraction,
 * no fast math.
 * ============================================================================================ */
#include "recovery_oracle.h"

#include <math.h>
#include <stdlib.h>
#include <string.h>

#include "shared_stream.h"

static inline double u53(uint32_t hi, uint32_t lo) {
    uint64_t v = (((uint64_t)hi << 32) | (uint64_t)lo) >> 11;
    return (double)v * 0x1p-53;
}

uint32_t ss_recovery_slot(double u_c, uint32_t n_free) {
    uint32_t k = (uint32_t)(u_c * (double)n_free);
    return k < n_free - 1u ? k : n_free - 1u;
}

int ss_recovery_draw(uint64_t seed, uint64_t step, uint64_t particle, double p, const uint32_t* free_cells, uint32_t n_free,
                     uint64_t grid_h, double pos_x, double pos_y, double res, float* out_xyt) {
    uint32_t key[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)};
    uint32_t ca[4] = {(uint32_t)particle, (uint32_t)step, (uint32_t)(step >> 32), 4u};
    uint32_t cb[4] = {(uint32_t)particle, (uint32_t)step, (uint32_t)(step >> 32), 5u};
    uint32_t cc[4] = {(uint32_t)particle, (uint32_t)step, (uint32_t)(step >> 32), 6u};
    uint32_t a[4], b[4], c[4];
    ss_philox4x32_10(ca, key, a);
    if (!(u53(a[0], a[1]) < p)) return 0;
    uint32_t cell = free_cells[ss_recovery_slot(u53(a[2], a[3]), n_free)];
    ss_philox4x32_10(cb, key, b);
    ss_philox4x32_10(cc, key, c);
    double col = (double)(cell % grid_h), row = (double)(cell / grid_h);
    out_xyt[0] = (float)(pos_x + (col + u53(b[0], b[1])) * res);
    out_xyt[1] = (float)(pos_y + (row + u53(b[2], b[3])) * res);
    out_xyt[2] = (float)(-0x1.921fb54442d18p+1 + u53(c[0], c[1]) * 0x1.921fb54442d18p+2);
    return 1;
}

void ss_fill_recovery_draws(uint64_t seed, uint64_t step, uint64_t first, uint64_t count, double p, const uint32_t* free_cells,
                            uint32_t n_free, uint64_t grid_h, double pos_x, double pos_y, double res, uint8_t* inject,
                            float* out_xyt) {
    for (uint64_t i = 0; i < count; ++i)
        inject[i] = (uint8_t)ss_recovery_draw(seed, step, first + i, p, free_cells, n_free, grid_h, pos_x, pos_y, res,
                                              out_xyt + 3 * i);
}

double so_recovery_update(double sum, uint64_t n, double alpha_slow, double alpha_fast, double* w_slow, double* w_fast) {
    if (!isfinite(sum)) return 0.0;
    const double w_avg = sum / (double)n;
    *w_slow = *w_slow == 0.0 ? w_avg : *w_slow + alpha_slow * (w_avg - *w_slow);
    *w_fast = *w_fast == 0.0 ? w_avg : *w_fast + alpha_fast * (w_avg - *w_fast);
    if (!(*w_slow > 0.0)) return 0.0;
    const double p = 1.0 - *w_fast / *w_slow;
    return p > 0.0 ? p : 0.0;   /* (NaN -> 0) */
}

struct so_rec {
    struct so_loc* loc;
    uint64_t n, gh;
    double pos_x, pos_y, res;      /* the config's f32 values, widened */
    uint32_t* free_cells;          /* ascending cell indices with p < 0.5 */
    uint32_t n_free;
    uint64_t step;                 /* updates so far (the stream's step) */
    so_pose est;                   /* estimated_pose of the last update, recorded before any injection */
    int has_est;
    int on, last;                  /* recovery is on / ran in the last update */
    double alpha_slow, alpha_fast, w_slow, w_fast, p;
    uint64_t seed, injected;
    double* raw;                   /* scratch: n raw weights */
    float* xyt;                    /* scratch: n poses */
};

struct so_rec* so_rec_create(float pos_x, float pos_y, float resolution, uint64_t gw, uint64_t gh, uint64_t n_particles,
                             int kind, float sigma, float z_rand, float occupied_above, const double* map) {
    struct so_rec* r = (struct so_rec*)calloc(1, sizeof(*r));
    if (!r) return NULL;
    r->loc = so_loc_create(pos_x, pos_y, resolution, gw, gh, n_particles, kind, sigma, z_rand, occupied_above, map);
    const uint64_t cells = gw * gh;
    r->free_cells = (uint32_t*)malloc((cells ? cells : 1) * sizeof(uint32_t));
    r->raw = (double*)malloc((n_particles ? n_particles : 1) * sizeof(double));
    r->xyt = (float*)malloc((n_particles ? n_particles : 1) * 3 * sizeof(float));
    if (!r->loc || !r->free_cells || !r->raw || !r->xyt) { so_rec_destroy(r); return NULL; }
    r->n = n_particles; r->gh = gh;
    r->pos_x = (double)pos_x; r->pos_y = (double)pos_y; r->res = (double)resolution;
    for (uint64_t c = 0; c < cells; ++c)
        if (map[c] < 0.5) r->free_cells[r->n_free++] = (uint32_t)c;
    return r;
}

void so_rec_destroy(struct so_rec* r) {
    if (!r) return;
    so_loc_destroy(r->loc);
    free(r->free_cells); free(r->raw); free(r->xyt);
    free(r);
}

struct so_loc* so_rec_loc(struct so_rec* r) { return r->loc; }

uint64_t so_rec_free_cells(const struct so_rec* r, uint32_t* out) {
    if (out) memcpy(out, r->free_cells, (size_t)r->n_free * sizeof(uint32_t));
    return r->n_free;
}

void so_rec_set_recovery(struct so_rec* r, double alpha_slow, double alpha_fast, uint64_t seed) {
    r->on = alpha_fast > 0.0;
    r->alpha_slow = alpha_slow; r->alpha_fast = alpha_fast; r->seed = seed;
    r->w_slow = r->w_fast = r->p = 0.0;
    r->injected = 0;
    r->last = 0;
}

int so_rec_update(struct so_rec* r, const double* angle, const double* dist, const uint8_t* valid, uint64_t nb, float dl,
                  float dr, float wheel, const double* z, double u01) {
    const uint64_t step = r->step++;
    const int rc = so_loc_update(r->loc, angle, dist, valid, nb, dl, dr, wheel, z, u01);
    if (rc < 0) return rc;
    /* estimated_pose, slam.rs:77-81: the resampled pose of max_particle, before anything is injected */
    r->est = so_loc_estimated_pose(r->loc);
    r->has_est = 1;
    r->p = 0.0;
    r->injected = 0;
    r->last = r->on;
    if (!r->on) return rc;
    so_loc_get_weights(r->loc, NULL, r->raw);   /* the raw weights resampling used (the device's under an override) */
    double sum = 0.0;
    for (uint64_t i = 0; i < r->n; ++i) sum += r->raw[i];
    r->p = so_recovery_update(sum, r->n, r->alpha_slow, r->alpha_fast, &r->w_slow, &r->w_fast);
    if (!(r->p > 0.0)) return rc;
    so_loc_get_poses(r->loc, r->xyt);
    for (uint64_t m = 0; m < r->n; ++m)
        r->injected += (uint64_t)ss_recovery_draw(r->seed, step, m, r->p, r->free_cells, r->n_free, r->gh, r->pos_x,
                                                  r->pos_y, r->res, r->xyt + 3 * m);
    so_loc_set_poses(r->loc, r->xyt);
    return rc;
}

void so_rec_state(const struct so_rec* r, double* out3, uint64_t* injected) {
    out3[0] = r->last ? r->w_slow : 0.0;
    out3[1] = r->last ? r->w_fast : 0.0;
    out3[2] = r->last ? r->p : 0.0;
    if (injected) *injected = r->last ? r->injected : 0;
}

so_pose so_rec_estimated_pose(const struct so_rec* r) { return r->has_est ? r->est : so_loc_estimated_pose(r->loc); }
