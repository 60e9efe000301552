/* TEST INFRASTRUCTURE ONLY -- CPU oracle of the localiser's recovery (augmented MCL, slamrs_gpu_set_recovery),
 * see recovery_oracle.c. */
#ifndef SLAMRS_RECOVERY_ORACLE_H
#define SLAMRS_RECOVERY_ORACLE_H
#include <stdint.h>
#include "loc_oracle.h"
#ifdef __cplusplus
extern "C" {
#endif

/* The recovery draw, counters (particle, step lo, step hi, 4 / 5 / 6) of the shared stream: decision
 * u_d = u53(a0, a1) < p; cell free_cells[ss_recovery_slot(u53(a2, a3), n_free)] (index row * grid_h + column);
 * x = (float)(pos_x + (col + u53(b0, b1)) * res), y = (float)(pos_y + (row + u53(b2, b3)) * res),
 * theta = (float)(-pi + u53(c0, c1) * 2pi). Returns 1 and writes out_xyt when the particle is replaced, else 0. */
uint32_t ss_recovery_slot(double u_c, uint32_t n_free);
int ss_recovery_draw(uint64_t seed, uint64_t step, uint64_t particle, double p, const uint32_t* free_cells, uint32_t n_free,
                     uint64_t grid_h, double pos_x, double pos_y, double res, float* out_xyt);
void ss_fill_recovery_draws(uint64_t seed, uint64_t step, uint64_t first, uint64_t count, double p, const uint32_t* free_cells,
                            uint32_t n_free, uint64_t grid_h, double pos_x, double pos_y, double res, uint8_t* inject,
                            float* out_xyt);
/* one step of the averages on the raw-weight sum of n particles; returns p */
double so_recovery_update(double sum, uint64_t n, double alpha_slow, double alpha_fast, double* w_slow, double* w_fast);

/* A localiser oracle (loc_oracle.c) with recovery behind its resampling. The so_loc_* accessors apply to
 * so_rec_loc(r); update and the estimate go through so_rec_update / so_rec_estimated_pose. */
struct so_rec;
struct so_rec* so_rec_create(float pos_x, float pos_y, float resolution, uint64_t gw, uint64_t gh, uint64_t n_particles,
                             int kind, float sigma, float z_rand, float occupied_above, const double* map);
void so_rec_destroy(struct so_rec* r);
struct so_loc* so_rec_loc(struct so_rec* r);
uint64_t so_rec_free_cells(const struct so_rec* r, uint32_t* out);
/* alpha_fast > 0: on (with the stream keyed by seed), else off; resets the averages */
void so_rec_set_recovery(struct so_rec* r, double alpha_slow, double alpha_fast, uint64_t seed);
int so_rec_update(struct so_rec* r, const double* angle, const double* dist, const uint8_t* valid, uint64_t nb, float dl,
                  float dr, float wheel, const double* z, double u01);
/* {w_slow, w_fast, p} and the injected count of the last update; all zero when it ran without recovery */
void so_rec_state(const struct so_rec* r, double* out3, uint64_t* injected);
so_pose so_rec_estimated_pose(const struct so_rec* r);

#ifdef __cplusplus
}
#endif
#endif
