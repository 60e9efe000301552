// Device helpers shared by the kernel translation units (kernels_*.cu): streaming 128/256-bit
// accesses and deterministic block-wide prefix sums.
#pragma once
#include "kernels.cuh"
#include "shared_stream.cuh"
#include <cooperative_groups.h>

namespace slamrs {

// Programmatic dependent launch (sm_90+): a kernel launched with launch_pdl() may become resident while the kernel in
// front of it in the stream still runs -- once that one has let its dependents go (pdl_launch_dependents) -- and must
// not touch anything the stream order protects before pdl_wait() returns (the prerequisite grid has completed and its
// writes are visible). Without the launch attribute both are no-ops. Takes the launch latency and the ramp of the
// short kernels of the step (motion -> likelihood -> weights -> indices) out of the critical path.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}


namespace cg = cooperative_groups;


__device__ __forceinline__ uint4 ld_stream_v4(const uint4* p) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p));
    return r;
}
__device__ __forceinline__ void st_stream_v4(uint4* p, const uint4& v) {
    asm volatile("st.global.L1::no_allocate.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z),
                 "r"(v.w)
                 : "memory");
}

// exclusive prefix sum of one uint32 per thread over a 1024-thread CTA (warp shuffles + one
// shared array of 32 warp totals). Returns the exclusive prefix; *total gets the CTA sum.
__device__ __forceinline__ uint32_t block_excl_scan_u32(uint32_t v, uint32_t* warp_tot /*[33]*/, uint32_t* total) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    uint32_t inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
    }
    __syncthreads();  // protect warp_tot reuse across calls
    if (lane == 31) warp_tot[wid] = inc;
    __syncthreads();
    if (wid == 0) {
        uint32_t w = lane < nw ? warp_tot[lane] : 0u;
        uint32_t winc = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, winc, o);
            if (lane >= o) winc += t;
        }
        warp_tot[lane] = winc - w;  // exclusive warp offsets
        if (lane == 31) warp_tot[32] = winc;
    }
    __syncthreads();
    *total = warp_tot[32];
    return warp_tot[wid] + inc - v;
}

// same for doubles (fixed combination order => deterministic)
__device__ __forceinline__ double block_excl_scan_f64(double v, double* warp_tot /*[33]*/, double* total) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    double inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const double t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc = __dadd_rn(t, inc);
    }
    __syncthreads();
    if (lane == 31) warp_tot[wid] = inc;
    __syncthreads();
    if (wid == 0) {
        const double w = lane < nw ? warp_tot[lane] : 0.0;
        double winc = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const double t = __shfl_up_sync(0xffffffffu, winc, o);
            if (lane >= o) winc = __dadd_rn(t, winc);
        }
        const double excl = __shfl_up_sync(0xffffffffu, winc, 1);
        warp_tot[lane] = lane == 0 ? 0.0 : excl;
        if (lane == 31) warp_tot[32] = winc;
    }
    __syncthreads();
    *total = warp_tot[32];
    // exclusive prefix of this thread = warp offset + (inclusive - own) within the warp
    const double within = __shfl_up_sync(0xffffffffu, inc, 1);
    return lane == 0 ? warp_tot[wid] : __dadd_rn(warp_tot[wid], within);
}

// The motion log-density Odometry::probabiliy_of (robot.rs:152-167) of a move from (ox, oy, otheta) to (nx, ny, ntheta)
__device__ __forceinline__ double motion_log_density(const OdomModel& od, float ox, float oy, float otheta, float nx,
                                                     float ny, float ntheta) {
    const float dx = __fsub_rn(ox, nx), dy = __fsub_rn(oy, ny);
    const float moved = __fsqrt_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)));
    const double ad = angle_diff((double)otheta, (double)ntheta);
    return __dadd_rn(log(normal_pdf((double)moved, od.mean_c, od.std_c)), log(normal_pdf(ad, od.mean_t, od.std_t)));
}

// Odometry::sample (robot.rs:170-183) and the motion log-density Odometry::probabiliy_of (robot.rs:152-167) of local
// particle p (global index gp) moved from pose_cur: the draws come from z_draws (RNG_CALLER) or the shared stream.
// Returns the new pose and, in `weight`, the log-density (slot is left to the caller).
__device__ __forceinline__ ParticleResult motion_step(const OdomModel& od, const float* __restrict__ pose_cur, uint32_t p,
                                                      uint32_t gp, const double* __restrict__ z_draws, uint64_t seed,
                                                      uint64_t step) {
    const float ox = pose_cur[3 * p], oy = pose_cur[3 * p + 1], otheta = pose_cur[3 * p + 2];
    // Odometry::sample. statrs: sample = mean + std_dev * z.
    double z1, z2;
    if (z_draws) {
        z1 = z_draws[2 * (size_t)gp];
        z2 = z_draws[2 * (size_t)gp + 1];
    } else {
        slamrs_stream::motion_normals(seed, step, gp, &z1, &z2);
    }
    const float center_distance = (float)__dadd_rn(od.mean_c, __dmul_rn(od.std_c, z1));
    const float ntheta = __fadd_rn(otheta, (float)__dadd_rn(od.mean_t, __dmul_rn(od.std_t, z2)));
    float sn, cs;
    slamrs_libm::sincosf_exact(ntheta, &sn, &cs);
    const float nx = __fadd_rn(ox, __fmul_rn(cs, center_distance));
    const float ny = __fadd_rn(oy, __fmul_rn(sn, center_distance));
    ParticleResult r;
    r.weight = motion_log_density(od, ox, oy, otheta, nx, ny, ntheta);   // Odometry::probabiliy_of(old, new)
    r.x = nx; r.y = ny; r.theta = ntheta;
    r.slot = -1;
    return r;
}

// Compacts the (angle, distance) pairs of the VALID beams among [b_begin, b_end), in beam order, into out[0..) and
// returns their number to every thread. Only valid measurements contribute to Map::probability_of (map.rs:117-119);
// one coalesced 8-byte load per beam replaces the dependent valid[] -> angle[], dist[] loads. Called by every
// thread of a 128-thread CTA.
__device__ __forceinline__ uint32_t block_compact_valid_beams(const ScanDevice& scan, uint32_t b_begin, uint32_t b_end,
                                                              float2* out) {
    __shared__ uint32_t s_cnt[4];
    __shared__ uint32_t s_base;
    if (threadIdx.x == 0) s_base = 0u;
    __syncthreads();
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    for (uint32_t b0 = b_begin; b0 < b_end; b0 += 128u) {
        const uint32_t b = b0 + threadIdx.x;
        const bool v = b < b_end && scan.valid[b] != 0;
        const unsigned m = __ballot_sync(0xffffffffu, v);
        if (lane == 0) s_cnt[wid] = __popc(m);
        __syncthreads();
        uint32_t off = s_base;
        for (int w = 0; w < wid; ++w) off += s_cnt[w];
        if (v) out[off + __popc(m & ((1u << lane) - 1u))] = make_float2(scan.angle[b], scan.dist[b]);
        __syncthreads();
        if (threadIdx.x == 0) s_base += s_cnt[0] + s_cnt[1] + s_cnt[2] + s_cnt[3];
        __syncthreads();
    }
    return s_base;
}

struct alignas(32) V8 {
    uint4 a, b;
};
// 256-bit global accesses (sm_100: ld/st.global.v8.b32). Streaming: no L1 allocation.
__device__ __forceinline__ V8 ld_stream_v8(const V8* p) {
    V8 r;
    asm volatile("ld.global.nc.L1::no_allocate.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r.a.x), "=r"(r.a.y), "=r"(r.a.z), "=r"(r.a.w), "=r"(r.b.x), "=r"(r.b.y), "=r"(r.b.z), "=r"(r.b.w)
                 : "l"(p));
    return r;
}
__device__ __forceinline__ void st_stream_v8(V8* p, const V8& v) {
    asm volatile("st.global.L1::no_allocate.v8.u32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "r"(v.a.x), "r"(v.a.y),
                 "r"(v.a.z), "r"(v.a.w), "r"(v.b.x), "r"(v.b.y), "r"(v.b.z), "r"(v.b.w)
                 : "memory");
}

}  // namespace slamrs
