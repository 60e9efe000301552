/* ============================================================================================
 * TEST INFRASTRUCTURE ONLY -- CPU oracle of the localiser's pose clusters (slamrs_gpu_pose_clusters;
 * ROS AMCL's pf_cluster_stats with the heading wrapping around): the bins are kld_oracle.c's
 * so_kld_bin, the occupied bins are sorted, and a sequential union-find joins each one to its
 * occupied neighbours. The moments are computed from these labels in cluster_oracle.py.
 * ============================================================================================ */
#include "cluster_oracle.h"

#include <math.h>
#include <stdlib.h>

#include "kld_oracle.h"

static int cmp_u64(const void* a, const void* b) {
    const uint64_t x = *(const uint64_t*)a, y = *(const uint64_t*)b;
    return (x > y) - (x < y);
}

/* index of bin b among the n sorted occupied bins, or n when it is not occupied */
static uint64_t find_bin(const uint64_t* occ, uint64_t n, uint64_t b) {
    uint64_t lo = 0, hi = n;
    while (lo < hi) {
        const uint64_t mid = lo + (hi - lo) / 2;
        if (occ[mid] < b) lo = mid + 1;
        else hi = mid;
    }
    return lo < n && occ[lo] == b ? lo : n;
}

static uint64_t root_of(uint64_t* parent, uint64_t x) {
    while (parent[x] != x) x = parent[x];
    return x;
}

typedef struct { uint64_t label, count; } ranked;

static int cmp_ranked(const void* a, const void* b) {
    const ranked* x = (const ranked*)a;
    const ranked* y = (const ranked*)b;
    if (x->count != y->count) return x->count > y->count ? -1 : 1;
    return (x->label > y->label) - (x->label < y->label);
}

int so_pose_clusters(const float* xyt, uint64_t n, float pos_x, float pos_y, float res, uint64_t gw, uint64_t gh,
                     uint32_t bin_cells, uint32_t theta_bins, uint64_t* labels, uint64_t* out3, uint64_t* ranked_label,
                     uint64_t* ranked_count) {
    const uint64_t nbx = (gw + bin_cells - 1) / bin_cells, nby = (gh + bin_cells - 1) / bin_cells;
    const uint64_t off_grid = nbx * nby * theta_bins;
    uint64_t* bin = (uint64_t*)malloc((n ? n : 1) * sizeof(uint64_t));
    uint64_t* occ = (uint64_t*)malloc((n ? n : 1) * sizeof(uint64_t));
    uint64_t* parent = (uint64_t*)malloc((n ? n : 1) * sizeof(uint64_t));
    uint64_t* count = (uint64_t*)calloc(n ? n : 1, sizeof(uint64_t));
    ranked* rk = (ranked*)malloc((n ? n : 1) * sizeof(ranked));
    if (!bin || !occ || !parent || !count || !rk) {
        free(bin); free(occ); free(parent); free(count); free(rk);
        return -1;
    }
    /* bins (item 2, 3) */
    uint64_t n_excluded = 0, m = 0;
    for (uint64_t i = 0; i < n; ++i) {
        const float x = xyt[3 * i], y = xyt[3 * i + 1], t = xyt[3 * i + 2];
        uint64_t b = SO_CLUSTER_EXCLUDED;
        if (isfinite(x) && isfinite(y) && isfinite(t)) {
            b = so_kld_bin(x, y, t, pos_x, pos_y, res, gw, gh, bin_cells, theta_bins);
            if (b == off_grid) b = SO_CLUSTER_EXCLUDED;
        }
        bin[i] = b;
        if (b == SO_CLUSTER_EXCLUDED) ++n_excluded;
        else occ[m++] = b;
    }
    qsort(occ, m, sizeof(uint64_t), cmp_u64);
    uint64_t n_bins = 0;
    for (uint64_t j = 0; j < m; ++j)
        if (j == 0 || occ[j] != occ[j - 1]) occ[n_bins++] = occ[j];
    /* components (item 4): union of every occupied bin with each occupied neighbour, the smaller root kept */
    for (uint64_t r = 0; r < n_bins; ++r) parent[r] = r;
    for (uint64_t r = 0; r < n_bins; ++r) {
        const uint64_t b = occ[r], h = b % theta_bins, cell = b / theta_bins, bx = cell % nbx, by = cell / nbx;
        for (int dy = -1; dy <= 1; ++dy)
            for (int dx = -1; dx <= 1; ++dx)
                for (int dh = -1; dh <= 1; ++dh) {
                    const int64_t y2 = (int64_t)by + dy, x2 = (int64_t)bx + dx;
                    if (y2 < 0 || y2 >= (int64_t)nby || x2 < 0 || x2 >= (int64_t)nbx) continue;
                    const uint64_t h2 = (uint64_t)(((int64_t)h + dh + (int64_t)theta_bins) % (int64_t)theta_bins);
                    const uint64_t s = find_bin(occ, n_bins, ((uint64_t)y2 * nbx + (uint64_t)x2) * theta_bins + h2);
                    if (s == n_bins) continue;
                    const uint64_t a = root_of(parent, r), c = root_of(parent, s);
                    if (a < c) parent[c] = a;
                    else parent[a] = c;
                }
    }
    /* labels and counts (the root of a component is its smallest index, hence its smallest bin id) */
    uint64_t n_clusters = 0;
    for (uint64_t r = 0; r < n_bins; ++r) n_clusters += root_of(parent, r) == r;
    for (uint64_t i = 0; i < n; ++i) {
        if (bin[i] == SO_CLUSTER_EXCLUDED) { labels[i] = SO_CLUSTER_EXCLUDED; continue; }
        const uint64_t root = root_of(parent, find_bin(occ, n_bins, bin[i]));
        labels[i] = occ[root];
        ++count[root];
    }
    /* order (item 5) */
    uint64_t k = 0;
    for (uint64_t r = 0; r < n_bins; ++r)
        if (parent[r] == r) { rk[k].label = occ[r]; rk[k].count = count[r]; ++k; }
    qsort(rk, k, sizeof(ranked), cmp_ranked);
    for (uint64_t j = 0; j < k; ++j) { ranked_label[j] = rk[j].label; ranked_count[j] = rk[j].count; }
    out3[0] = n_excluded; out3[1] = n_bins; out3[2] = n_clusters;
    free(bin); free(occ); free(parent); free(count); free(rk);
    return 0;
}
