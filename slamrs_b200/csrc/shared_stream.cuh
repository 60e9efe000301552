// The shared seeded stream: motion-noise normals and the resample uniform.
//
// The reference draws from rand::thread_rng() (slamrs/common/src/robot.rs:173, two statrs
// Normal samples per particle) and rand::random::<f64>() (slamrs/slam/src/grid/particle.rs:84).
// Those are OS-seeded; here both come from one counter-based stream so that any two
// implementations given (seed, step, particle) consume identical bits:
//
//   bits    Philox4x32-10, key = (seed lo32, seed hi32)
//   motion  counter (particle, step lo32, step hi32, 0) -> x0..x3
//           u1 = (((x0:x1) >> 11) + 1) * 2^-53 in (0,1];  u2 = ((x2:x3) >> 11) * 2^-53 in [0,1)
//           r = sqrt(-2 dlog(u1));  z1 = r * dcos(2 pi u2)  (centre distance draw)
//                                   z2 = r * dsin(2 pi u2)  (heading draw)
//   uniform counter (0, step lo32, step hi32, 1) -> U = ((x0:x1) >> 11) * 2^-53
//   start   counter (particle, 0, 0, 2) and (particle, 0, 0, 3): uniform_pose
//   recover counter (particle, step lo32, step hi32, 4 / 5 / 6): recovery_draw
//
// dlog / dsincos2pi are fixed sequences of IEEE binary64 + - * / (explicit round-to-nearest
// intrinsics on the device, so no FMA contraction), which makes the stream bit-identical on
// CPU and GPU without uploading draws.
#pragma once
#include <stdint.h>
#include <math.h>

#if defined(__CUDACC__)
#define SS_HD __host__ __device__ __forceinline__
#else
#define SS_HD static inline
#endif

namespace slamrs_stream {

SS_HD double dmul(double a, double b) {
#if defined(__CUDA_ARCH__)
    return __dmul_rn(a, b);
#else
    return a * b;
#endif
}
SS_HD double dadd(double a, double b) {
#if defined(__CUDA_ARCH__)
    return __dadd_rn(a, b);
#else
    return a + b;
#endif
}
SS_HD double ddiv(double a, double b) {
#if defined(__CUDA_ARCH__)
    return __ddiv_rn(a, b);
#else
    return a / b;
#endif
}
SS_HD double dsqrt(double a) {
#if defined(__CUDA_ARCH__)
    return __dsqrt_rn(a);
#else
    return sqrt(a);
#endif
}

struct Words4 {
    uint32_t x[4];
};

SS_HD Words4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint64_t p0 = (uint64_t)0xD2511F53u * c0;
        const uint64_t p1 = (uint64_t)0xCD9E8D57u * c2;
        const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
        const uint32_t n1 = (uint32_t)p1;
        const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
        const uint32_t n3 = (uint32_t)p0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    Words4 w;
    w.x[0] = c0; w.x[1] = c1; w.x[2] = c2; w.x[3] = c3;
    return w;
}

SS_HD double bits_to_double(uint64_t b) {
#if defined(__CUDA_ARCH__)
    return __longlong_as_double((long long)b);
#else
    double d;
    __builtin_memcpy(&d, &b, 8);
    return d;
#endif
}
SS_HD uint64_t double_to_bits(double d) {
#if defined(__CUDA_ARCH__)
    return (uint64_t)__double_as_longlong(d);
#else
    uint64_t b;
    __builtin_memcpy(&b, &d, 8);
    return b;
#endif
}

// ln(x) for positive normal x: x = m 2^e with m in [sqrt(1/2), sqrt(2)),
// s = (m-1)/(m+1), ln m = 2 s (1 + s^2/3 + s^4/5 + ... + s^22/23)
SS_HD double dlog(double x) {
    uint64_t b = double_to_bits(x);
    int e = (int)((b >> 52) & 0x7ff) - 1023;
    b = (b & 0x000fffffffffffffULL) | 0x3ff0000000000000ULL;
    double m = bits_to_double(b);
    if (m > 0x1.6a09e667f3bcdp+0) {
        m = dmul(m, 0.5);
        e += 1;
    }
    const double s = ddiv(dadd(m, -1.0), dadd(m, 1.0));
    const double z = dmul(s, s);
    const double c[12] = {
        0x1.0000000000000p+0, 0x1.5555555555555p-2, 0x1.999999999999ap-3, 0x1.2492492492492p-3,
        0x1.c71c71c71c71cp-4, 0x1.745d1745d1746p-4, 0x1.3b13b13b13b14p-4, 0x1.1111111111111p-4,
        0x1.e1e1e1e1e1e1ep-5, 0x1.af286bca1af28p-5, 0x1.8618618618618p-5, 0x1.642c8590b2164p-5};
    double p = c[11];
#pragma unroll
    for (int k = 10; k >= 0; --k) p = dadd(dmul(p, z), c[k]);
    const double lnm = dmul(dmul(2.0, s), p);
    return dadd(dmul((double)e, 0x1.62e42fefa39efp-1), lnm);
}

// sin/cos of 2 pi u, u in [0,1): quadrant k = floor(4u), t = (4u - k) pi/2, Taylor to t^25 / t^24
SS_HD void dsincos2pi(double u, double* s_out, double* c_out) {
    const double q = dmul(u, 4.0);
    const int k = (int)q;
    const double f = dadd(q, -(double)k);
    const double t = dmul(f, 0x1.921fb54442d18p+0);
    const double t2 = dmul(t, t);
    const double sc[13] = {
        0x1.0000000000000p+0,   -0x1.5555555555555p-3,  0x1.1111111111111p-7,
        -0x1.a01a01a01a01ap-13, 0x1.71de3a556c734p-19,  -0x1.ae64567f544e4p-26,
        0x1.6124613a86d09p-33,  -0x1.ae7f3e733b81fp-41, 0x1.952c77030ad4ap-49,
        -0x1.2f49b46814157p-57, 0x1.71b8ef6dcf572p-66,  -0x1.761b41316381ap-75,
        0x1.3f3ccdd165fa9p-84};
    const double cc[13] = {
        0x1.0000000000000p+0,   -0x1.0000000000000p-1,  0x1.5555555555555p-5,
        -0x1.6c16c16c16c17p-10, 0x1.a01a01a01a01ap-16,  -0x1.27e4fb7789f5cp-22,
        0x1.1eed8eff8d898p-29,  -0x1.93974a8c07c9dp-37, 0x1.ae7f3e733b81fp-45,
        -0x1.6827863b97d97p-53, 0x1.e542ba4020225p-62,  -0x1.0ce396db7f853p-70,
        0x1.f2cf01972f578p-80};
    double ps = sc[12], pc = cc[12];
#pragma unroll
    for (int i = 11; i >= 0; --i) {
        ps = dadd(dmul(ps, t2), sc[i]);
        pc = dadd(dmul(pc, t2), cc[i]);
    }
    const double st = dmul(ps, t), ct = pc;
    switch (k & 3) {
        case 0: *s_out = st;  *c_out = ct;  break;
        case 1: *s_out = ct;  *c_out = -st; break;
        case 2: *s_out = -st; *c_out = -ct; break;
        default: *s_out = -ct; *c_out = st; break;
    }
}

SS_HD double u53(uint32_t hi, uint32_t lo) {
    const uint64_t v = (((uint64_t)hi << 32) | (uint64_t)lo) >> 11;
    return dmul((double)v, 0x1p-53);
}

SS_HD void motion_normals(uint64_t seed, uint64_t step, uint32_t particle, double* z1, double* z2) {
    const Words4 w = philox4x32_10(particle, (uint32_t)step, (uint32_t)(step >> 32), 0u, (uint32_t)seed,
                                   (uint32_t)(seed >> 32));
    const uint64_t v1 = ((((uint64_t)w.x[0] << 32) | (uint64_t)w.x[1]) >> 11) + 1;
    const double u1 = dmul((double)v1, 0x1p-53);
    const double u2 = u53(w.x[2], w.x[3]);
    const double r = dsqrt(dmul(-2.0, dlog(u1)));
    double s, c;
    dsincos2pi(u2, &s, &c);
    *z1 = dmul(r, c);
    *z2 = dmul(r, s);
}

SS_HD double resample_uniform(uint64_t seed, uint64_t step) {
    const Words4 w = philox4x32_10(0u, (uint32_t)step, (uint32_t)(step >> 32), 1u, (uint32_t)seed,
                                   (uint32_t)(seed >> 32));
    return u53(w.x[0], w.x[1]);
}

// Start pose of `particle` for a uniform initialisation over the box [x0, x1) x [y0, y1), heading in
// [-pi, pi): three 53-bit uniforms from the stream's own counter domains (2: position, 3: heading)
SS_HD void uniform_pose(uint64_t seed, uint32_t particle, double x0, double y0, double x1, double y1, float* px, float* py,
                        float* ptheta) {
    const Words4 a = philox4x32_10(particle, 0u, 0u, 2u, (uint32_t)seed, (uint32_t)(seed >> 32));
    const Words4 b = philox4x32_10(particle, 0u, 0u, 3u, (uint32_t)seed, (uint32_t)(seed >> 32));
    *px = (float)dadd(x0, dmul(u53(a.x[0], a.x[1]), dadd(x1, -x0)));
    *py = (float)dadd(y0, dmul(u53(a.x[2], a.x[3]), dadd(y1, -y0)));
    *ptheta = (float)dadd(-0x1.921fb54442d18p+1, dmul(u53(b.x[0], b.x[1]), 0x1.921fb54442d18p+2));
}

// Augmented-MCL recovery (slamrs_gpu_set_recovery). The averages of the raw weights, from the step's weight sum `sum`
// over n particles: w_avg = sum / n; w = (w == 0) ? w_avg : w + alpha (w_avg - w) for both averages; the share of
// particles to replace is p = max(0, 1 - w_fast / w_slow) (0 when w_slow is not positive, and for NaN). A sum that
// is not finite leaves both averages as they are and gives p = 0.
SS_HD double recovery_update(double sum, uint32_t n, double alpha_slow, double alpha_fast, double* w_slow, double* w_fast) {
    if (!isfinite(sum)) return 0.0;
    const double w_avg = ddiv(sum, (double)n);
    *w_slow = *w_slow == 0.0 ? w_avg : dadd(*w_slow, dmul(alpha_slow, dadd(w_avg, -*w_slow)));
    *w_fast = *w_fast == 0.0 ? w_avg : dadd(*w_fast, dmul(alpha_fast, dadd(w_avg, -*w_fast)));
    if (!(*w_slow > 0.0)) return 0.0;
    const double p = dadd(1.0, -ddiv(*w_fast, *w_slow));
    return p > 0.0 ? p : 0.0;
}
// Entry of the free-cell list that the cell uniform u_c in [0, 1) selects. (In round-to-nearest the product stays
// below n_free for every u_c the stream yields; the clamp keeps the index in range regardless.)
SS_HD uint32_t recovery_slot(double u_c, uint32_t n_free) {
    const uint32_t k = (uint32_t)dmul(u_c, (double)n_free);
    return k < n_free - 1u ? k : n_free - 1u;
}
// Is new particle `particle` of step `step` replaced (u_d < p), and by which pose: a cell drawn from the ascending
// list of free cells (index row * grid_h + column), a position uniform inside that cell and a heading in
// [-pi, pi) as uniform_pose draws it. Counter domains 4 (u_d, u_c), 5 (u_x, u_y) and 6 (u_t), keyed by the step;
// pos_x, pos_y and res are the config's f32 values widened. The poses of other particles are not touched.
SS_HD bool recovery_draw(uint64_t seed, uint64_t step, uint32_t particle, double p, const uint32_t* free_cells,
                         uint32_t n_free, uint32_t grid_h, double pos_x, double pos_y, double res, float* px, float* py,
                         float* ptheta) {
    const uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32), s0 = (uint32_t)step, s1 = (uint32_t)(step >> 32);
    const Words4 a = philox4x32_10(particle, s0, s1, 4u, k0, k1);
    if (!(u53(a.x[0], a.x[1]) < p)) return false;
    const uint32_t cell = free_cells[recovery_slot(u53(a.x[2], a.x[3]), n_free)];
    const Words4 b = philox4x32_10(particle, s0, s1, 5u, k0, k1);
    const Words4 c = philox4x32_10(particle, s0, s1, 6u, k0, k1);
    const double col = (double)(cell % grid_h), row = (double)(cell / grid_h);
    *px = (float)dadd(pos_x, dmul(dadd(col, u53(b.x[0], b.x[1])), res));
    *py = (float)dadd(pos_y, dmul(dadd(row, u53(b.x[2], b.x[3])), res));
    *ptheta = (float)dadd(-0x1.921fb54442d18p+1, dmul(u53(c.x[0], c.x[1]), 0x1.921fb54442d18p+2));
    return true;
}

}  // namespace slamrs_stream
