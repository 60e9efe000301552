/* TEST INFRASTRUCTURE ONLY -- CPU oracle of the localiser's KLD-sampling (adaptive population, slamrs_gpu_set_kld),
 * see kld_oracle.c. */
#ifndef SLAMRS_KLD_ORACLE_H
#define SLAMRS_KLD_ORACLE_H
#include <stdint.h>
#include "slam_oracle.h"
#ifdef __cplusplus
extern "C" {
#endif

/* The bin of a pose: cell (world_to_grid, is_valid, `as usize`) coarsened to bin_cells x bin_cells, times theta_bins
 * headings (t = fmod(theta, 2pi) + 2pi if negative; bin min(theta_bins - 1, (t * theta_bins) / 2pi) for 0 <= t < 2pi,
 * else 0). Every pose off the grid is in bin nbx * nby * theta_bins, nbx = ceil(gw / bin_cells). */
uint64_t so_kld_bin(float x, float y, float theta, float pos_x, float pos_y, float res, uint64_t gw, uint64_t gh,
                    uint32_t bin_cells, uint32_t theta_bins);
/* distinct bins of n poses {x, y, theta} */
uint64_t so_kld_count(const float* xyt, uint64_t n, float pos_x, float pos_y, float res, uint64_t gw, uint64_t gh,
                      uint32_t bin_cells, uint32_t theta_bins);
/* AMCL's pf_resample_limit for k bins, n_min for k <= 1 */
uint64_t so_kld_bound(uint64_t k, uint64_t n_min, uint64_t n_max, double err, double z);
/* so_resample_fold with m draws from the n weights: thresholds r = U * 1.0 / m, u = r + (j - 1) * 1.0 / m; the walk
 * over the n running sums and its clamp at n - 1 unchanged. idx receives m entries. Returns 1 when it clamped. */
int so_resample_fold_m(const double* raw, uint64_t n, uint64_t m, double u01, double* norm, uint64_t* idx,
                       uint64_t* max_particle);

/* The localiser update with a variable population (capacity n_particles): loc_oracle.c's step over the N_t poses of
 * the current generation, M = N_{t+1} draws (KLD-sampling on) or the capacity (off), the estimate at new particle
 * floor(max_particle * M / N_t), then recovery_oracle.c's recovery over the M new particles. */
struct so_kld;
struct so_kld* so_kld_create(float pos_x, float pos_y, float resolution, uint64_t gw, uint64_t gh, uint64_t n_particles,
                             int kind, float sigma, float z_rand, float occupied_above, const double* map);
void so_kld_destroy(struct so_kld* s);
/* on = 0: off (the next update draws the capacity) */
void so_kld_set_kld(struct so_kld* s, int on, uint64_t n_min, uint64_t n_max, double err, double z, uint32_t bin_cells,
                    uint32_t theta_bins);
/* alpha_fast > 0: on (stream keyed by seed), else off; resets the averages */
void so_kld_set_recovery(struct so_kld* s, double alpha_slow, double alpha_fast, uint64_t seed);
/* resample the next update on these N_t raw weights (the device's) */
void so_kld_set_weight_override(struct so_kld* s, const double* raw);
int so_kld_update(struct so_kld* s, const double* angle, const double* dist, const uint8_t* valid, uint64_t nb, float dl,
                  float dr, float wheel, const double* z, double u01);
uint64_t so_kld_population(const struct so_kld* s);
/* {N_t, k, M} of the last update; all zero when it ran without KLD-sampling */
void so_kld_state(const struct so_kld* s, uint64_t* out3);
void so_kld_recovery_state(const struct so_kld* s, double* out3, uint64_t* injected);
void so_kld_get_poses(const struct so_kld* s, float* out_xyt);      /* N entries */
void so_kld_set_poses(struct so_kld* s, const float* xyt);          /* N entries */
void so_kld_get_weights(const struct so_kld* s, double* norm, double* raw);   /* N_t entries each */
void so_kld_get_own_raw(const struct so_kld* s, double* out);                 /* N_t entries */
void so_kld_get_indices(const struct so_kld* s, uint64_t* idx);               /* M entries */
uint64_t so_kld_max_particle(const struct so_kld* s);
so_pose so_kld_estimated_pose(const struct so_kld* s);

#ifdef __cplusplus
}
#endif
#endif
