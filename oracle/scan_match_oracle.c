/* ============================================================================================
 * TEST INFRASTRUCTURE ONLY -- CPU oracle of scan-matching pose refinement (not in the reference: the slam.rs:60
 * TODO; the project's definition is DESIGN.md section 12). An integer score on the particle's pre-update hit
 * counters and a hill climb on it, so that the device's k_scan_match can be checked bit for bit.
 *
 * sm_update is so_update (GridMapSlam::update, slam.rs:46-75) with the climb between Odometry::sample and
 * Map::probability_of. It needs slam_oracle.c's map storage, endpoint, likelihood, integration and clone code,
 * which are static there, so this file includes slam_oracle.c and is compiled into a library of its own
 * (oracle/scan_match_oracle.py), with the flags of oracle/Makefile. The library works on handles that
 * liboracle.so's so_create / so_create_ex made: both are compiled from the same slam_oracle.c with the same flags,
 * so struct so_slam is the same in both, and both allocate with the C library's malloc. slam_oracle.c itself is
 * not changed: the default update stays so_update.
 * ============================================================================================ */
#include "slam_oracle.c"

/* the matcher's settings, as slamrs_gpu_scan_match */
typedef struct {
    uint32_t radius;      /* 0..2 cells */
    float step_xy;        /* metres */
    float step_theta;     /* radians */
    uint32_t levels;      /* 1..8 */
    uint32_t max_moves;   /* 1..1024 */
} sm_params;

/* occupied: log-odds of the saturated counters > 0, with the binary64 constants the device uses */
static inline int counters_occupied(uint16_t nf, uint16_t no) {
    return (double)nf * -0.8472978603872036 + (double)no * 2.1972245773362196 > 0.0;
}
static inline int map_cell_occupied(const struct so_map* m, uint64_t column, uint64_t row) {
    if (m->tiles) {
        const struct so_tile* t = m->tiles[tile_of(m, column, row)];
        return t ? counters_occupied(t->n_free[in_tile(column, row)], t->n_occ[in_tile(column, row)]) : 0;
    }
    const size_t idx = cell_index(m, column, row);
    return counters_occupied(m->n_free[idx], m->n_occ[idx]);
}
/* one beam: max((r+1)^2 - (dx^2 + dy^2)) over occupied cells at offsets in [-r, r]^2 of the endpoint's cell */
static uint32_t match_beam_score(const struct so_map* m, float ex, float ey, int r) {
    float gx, gy;
    world_to_grid(m, ex, ey, &gx, &gy);
    if (!is_valid(m, gx, gy)) return 0;
    const int64_t cx = (int64_t)f32_as_usize(gx), cy = (int64_t)f32_as_usize(gy);
    uint32_t best = 0;
    for (int dy = -r; dy <= r; ++dy)
        for (int dx = -r; dx <= r; ++dx) {
            const int64_t x = cx + dx, y = cy + dy;
            if (x < 0 || y < 0 || x >= (int64_t)m->gw || y >= (int64_t)m->gh) continue;
            if (!map_cell_occupied(m, (uint64_t)x, (uint64_t)y)) continue;
            const uint32_t v = (uint32_t)((r + 1) * (r + 1) - (dx * dx + dy * dy));
            if (v > best) best = v;
        }
    return best;
}
/* S(pose): the sum over the valid beams, endpoints as in map_log_probability_of */
static uint32_t match_score(const struct so_map* m, const double* angle, const double* dist, const uint8_t* valid,
                            uint64_t nb, so_pose pose, int r) {
    uint32_t sum = 0;
    for (uint64_t i = 0; i < nb; ++i) {
        if (!valid[i]) continue;
        float a = pose.theta + (float)angle[i];
        float ex = pose.x + cosf(a) * (float)dist[i];
        float ey = pose.y + sinf(a) * (float)dist[i];
        sum += match_beam_score(m, ex, ey, r);
    }
    return sum;
}
/* the hill climb from p; *moves and *scored receive its counts */
static so_pose match_climb(const sm_params* mp, const struct so_map* m, const double* angle, const double* dist,
                           const uint8_t* valid, uint64_t nb, so_pose p, uint32_t* moves, uint32_t* scored) {
    const int r = (int)mp->radius;
    uint32_t best = match_score(m, angle, dist, valid, nb, p, r);
    uint32_t mv = 0, sc = 1;
    for (uint32_t level = 0; level < mp->levels; ++level) {
        const float scale = ldexpf(1.0f, -(int)level);
        const float dxy = mp->step_xy * scale, dth = mp->step_theta * scale;
        while (mv < mp->max_moves) {
            so_pose cand[6];
            for (int k = 0; k < 6; ++k) cand[k] = p;
            cand[0].x = p.x + dxy; cand[1].x = p.x - dxy;
            cand[2].y = p.y + dxy; cand[3].y = p.y - dxy;
            cand[4].theta = p.theta + dth; cand[5].theta = p.theta - dth;
            int arg = 0;
            uint32_t top = 0;
            for (int k = 0; k < 6; ++k) {
                const uint32_t v = match_score(m, angle, dist, valid, nb, cand[k], r);
                sc++;
                if (k == 0 || v > top) { top = v; arg = k; }
            }
            if (top <= best) break;
            best = top;
            p = cand[arg];
            mv++;
        }
    }
    *moves = mv;
    *scored = sc;
    return p;
}


static int sm_params_ok(const struct so_slam* s, const sm_params* mp) {
    if (!s->track_counts && !s->sparse) return 0;   /* the score reads the hit counters */
    return mp->radius <= 2 && mp->step_xy > 0.0f && isfinite(mp->step_xy) && mp->step_theta > 0.0f &&
           isfinite(mp->step_theta) && mp->levels >= 1 && mp->levels <= 8 && mp->max_moves >= 1 && mp->max_moves <= 1024;
}

/* particle_step (the closure body of GridMapSlam::update, slam.rs:51-72) with the climb after the sample */
static void sm_particle_step(struct so_slam* s, uint64_t p, const double* angle, const double* dist, const uint8_t* valid,
                             uint64_t nb, const double od[4], const double* z, const sm_params* mp, uint32_t* moves,
                             uint32_t* scored) {
    so_pose initial = s->pose[p];
    so_pose np = so_odometry_sample(od, initial, z[2 * p], z[2 * p + 1]);
    struct so_map* m = &s->map[p];
    np = match_climb(mp, m, angle, dist, valid, nb, np, &moves[p], &scored[p]);
    double lw = map_log_probability_of(m, angle, dist, valid, nb, np) + so_odometry_log_prob(od, initial, np);
    map_integrate(s, m, angle, dist, valid, nb, np, (int64_t)p == s->trace_particle);
    s->pose[p] = np;
    s->raw_weight[p] = exp(lw);
}

/* so_update with scan matching; moves[p] and scored[p] receive each particle's climb counts. -2: bad settings, or a
 * handle without hit counters. Everything after the particle loop is so_update's, line for line. */
int sm_update(struct so_slam* s, const double* angle, const double* dist, const uint8_t* valid, uint64_t nb,
              float dl, float dr, float wheel, const double* z, double u01, const sm_params* mp, uint32_t* moves,
              uint32_t* scored) {
    if (!sm_params_ok(s, mp)) return -2;
    double od[4];
    so_odometry_new(dl, dr, wheel, od);
    s->trace_count = 0;
    const int64_t n = (int64_t)s->n;
#pragma omp parallel for schedule(dynamic, 1) num_threads(s->threads) if (s->threads > 1)
    for (int64_t p = 0; p < n; ++p) sm_particle_step(s, (uint64_t)p, angle, dist, valid, nb, od, z, mp, moves, scored);
    if (s->carry)   /* adaptive resampling: weights accumulate over the steps that did not resample */
        for (int64_t p = 0; p < n; ++p) s->raw_weight[p] = s->carry[p] * s->raw_weight[p];
    memcpy(s->own_raw, s->raw_weight, s->n * sizeof(double));
    if (s->weight_override) {   /* resample on the weights the device computed (see so_set_weight_override) */
        memcpy(s->raw_weight, s->weight_override, s->n * sizeof(double));
        s->weight_override = NULL;
    }
    /* normalize_weights, argmax, resample indices: particle.rs:40-56, 78-101 */
    s->clamped = so_resample_fold(s->raw_weight, s->n, u01, s->weight, NULL, s->last_idx, &s->max_particle);
    s->resampled = 1;
    if (s->adaptive_tau > 0.0) {
        /* NOT in the reference (which resamples after every scan, slam.rs:74): resample only when the effective
         * number of particles (particle.rs:59-65) drops below tau * N; otherwise every particle stays where it
         * is and carries its normalised weight into the next update. */
        double sq = 0.0;
        for (int64_t p = 0; p < n; ++p) sq += s->weight[p] * s->weight[p];
        if (!(1.0 / sq < s->adaptive_tau * (double)s->n)) {
            if (!s->carry) s->carry = (double*)malloc(s->n * sizeof(double));
            memcpy(s->carry, s->weight, s->n * sizeof(double));
            for (int64_t p = 0; p < n; ++p) s->last_idx[p] = (uint64_t)p;
            s->clamped = 0;
            s->resampled = 0;
            return 0;
        }
        free(s->carry);
        s->carry = NULL;
    }
    /* new generation: clone(old[i]) for every slot (deep copy of Pose + Map) */
    struct so_map* new_map = (struct so_map*)calloc(s->n, sizeof(struct so_map));
    so_pose* new_pose = (so_pose*)malloc(s->n * sizeof(so_pose));
    if (!new_map || !new_pose) { free(new_map); free(new_pose); return -1; }
    int fail = 0;
#pragma omp parallel for schedule(static) num_threads(s->threads) if (s->threads > 1)
    for (int64_t mm = 0; mm < n; ++mm) {
        if (map_alloc(&new_map[mm], s)) { fail = 1; continue; }
        map_copy(&new_map[mm], &s->map[s->last_idx[mm]]);
        new_pose[mm] = s->pose[s->last_idx[mm]];
    }
    if (fail) return -1;
    for (int64_t p = 0; p < n; ++p) map_free(&s->map[p]);
    free(s->map); free(s->pose);
    s->map = new_map; s->pose = new_pose;
    return s->clamped ? 1 : 0;
}

/* test hooks: S(pose) and the climb on particle p's current grid. -1 from sm_match_score: bad settings. */
int64_t sm_match_score(const struct so_slam* s, uint64_t particle, const double* angle, const double* dist,
                       const uint8_t* valid, uint64_t nb, so_pose pose, const sm_params* mp) {
    if (!sm_params_ok(s, mp)) return -1;
    return (int64_t)match_score(&s->map[particle], angle, dist, valid, nb, pose, (int)mp->radius);
}
int sm_match_climb(const struct so_slam* s, uint64_t particle, const double* angle, const double* dist,
                   const uint8_t* valid, uint64_t nb, so_pose pose, const sm_params* mp, so_pose* out_pose,
                   uint32_t out_moves_scored[2]) {
    if (!sm_params_ok(s, mp)) return -2;
    *out_pose = match_climb(mp, &s->map[particle], angle, dist, valid, nb, pose, &out_moves_scored[0],
                            &out_moves_scored[1]);
    return 0;
}
/* hand-built grids: particle p's hit counters, with the log-odds they stand for */
int sm_set_counts(struct so_slam* s, uint64_t particle, const uint16_t* n_free, const uint16_t* n_occ) {
    struct so_map* m = &s->map[particle];
    if (!m->tiles && !m->n_free) return -1;
    for (uint64_t row = 0; row < s->gh; ++row)
        for (uint64_t col = 0; col < s->gw; ++col) {
            const size_t src = cell_index(m, col, row);
            const double odds = s->l_prior + n_free[src] * s->l_free + n_occ[src] * s->l_occ;
            if (m->tiles) {
                if (!n_free[src] && !n_occ[src] && !m->tiles[tile_of(m, col, row)]) continue;
                struct so_tile* t = map_write_tile(m, col, row);
                t->odds[in_tile(col, row)] = odds;
                t->n_free[in_tile(col, row)] = n_free[src];
                t->n_occ[in_tile(col, row)] = n_occ[src];
            } else {
                m->odds[src] = odds;
                m->n_free[src] = n_free[src];
                m->n_occ[src] = n_occ[src];
            }
        }
    return 0;
}
/* 1 when sm_update accepts these settings on this handle */
int sm_check(const struct so_slam* s, const sm_params* mp) { return sm_params_ok(s, mp); }
