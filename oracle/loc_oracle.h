/* TEST INFRASTRUCTURE ONLY -- CPU oracle of the localiser (slamrs_gpu_create_localizer), see loc_oracle.c. */
#ifndef SLAMRS_LOC_ORACLE_H
#define SLAMRS_LOC_ORACLE_H
#include <stdint.h>
#include "slam_oracle.h"
#ifdef __cplusplus
extern "C" {
#endif

struct so_loc;
/* exact squared distance, in cells, from every cell to the nearest cell with p > occupied_above (index
 * row * gh + column); -1 everywhere when there is none. Returns the number of obstacle cells. */
int64_t so_loc_distance2(const double* map, uint64_t gw, uint64_t gh, double occupied_above, int64_t* out);
/* kind 0: beam endpoint (the reference's factor), 1: likelihood field */
struct so_loc* so_loc_create(float pos_x, float pos_y, float resolution, uint64_t gw, uint64_t gh, uint64_t n_particles,
                             int kind, float sigma, float z_rand, float occupied_above, const double* map);
void so_loc_destroy(struct so_loc* s);
void so_loc_terms(const struct so_loc* s, double* out);
double so_loc_outside(const struct so_loc* s);
void so_loc_set_adaptive_resampling(struct so_loc* s, double tau);
int so_loc_resampled(const struct so_loc* s);
void so_loc_set_weight_override(struct so_loc* s, const double* raw);
void so_loc_get_own_raw(const struct so_loc* s, double* out);
int so_loc_update(struct so_loc* s, const double* angle, const double* dist, const uint8_t* valid, uint64_t nb, float dl,
                  float dr, float wheel, const double* z, double u01);
void so_loc_get_poses(const struct so_loc* s, float* out_xyt);
void so_loc_set_poses(struct so_loc* s, const float* xyt);
void so_loc_get_weights(const struct so_loc* s, double* norm, double* raw);
void so_loc_get_indices(const struct so_loc* s, uint64_t* idx);
uint64_t so_loc_max_particle(const struct so_loc* s);
so_pose so_loc_estimated_pose(const struct so_loc* s);
double so_loc_effective_particles(const struct so_loc* s);
#ifdef __cplusplus
}
#endif
#endif
