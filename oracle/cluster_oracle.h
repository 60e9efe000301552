/* TEST INFRASTRUCTURE ONLY -- CPU oracle of the localiser's pose clusters (slamrs_gpu_pose_clusters), see
 * cluster_oracle.c. */
#ifndef SLAMRS_CLUSTER_ORACLE_H
#define SLAMRS_CLUSTER_ORACLE_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define SO_CLUSTER_EXCLUDED UINT64_MAX

/* The clusters of n poses {x, y, theta}: a pose with a non-finite component or off the grid is excluded; the others
 * fall into so_kld_bin's bins; occupied bins whose (bx, by) differ by at most 1 each and whose heading bins differ by
 * at most 1 modulo theta_bins are adjacent; a cluster is a connected component, labelled by its smallest bin id.
 * labels[i] = the label of pose i's cluster (SO_CLUSTER_EXCLUDED: excluded). out3 = {n_excluded, n_bins, n_clusters}.
 * ranked_label / ranked_count (n entries each, at least n_clusters are written) = every cluster by count descending,
 * then label ascending. Returns 0, or -1 when memory runs out. */
int so_pose_clusters(const float* xyt, uint64_t n, float pos_x, float pos_y, float res, uint64_t gw, uint64_t gh,
                     uint32_t bin_cells, uint32_t theta_bins, uint64_t* labels, uint64_t* out3, uint64_t* ranked_label,
                     uint64_t* ranked_count);

#ifdef __cplusplus
}
#endif
#endif
