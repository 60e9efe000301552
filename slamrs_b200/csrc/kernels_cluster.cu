// Pose clusters of the localiser's current generation (slamrs_gpu_pose_clusters; ROS AMCL's pf_cluster_stats), twelve
// launches chained by programmatic dependent launch:
//   k_cl_mark      one thread per pose: its bin (or none: excluded), the bin's bit in the bitmap
//   k_cl_words + k_loc_free_scan + k_cl_rank   ordered compaction of the bitmap: occupied bins by rank (= ascending
//                  bin id), the rank of a bin = prefix[b >> 5] + popc(word & below), parent[r] = r
//   k_cl_union     one thread per occupied bin: union-find over ranks with its occupied neighbours of larger id, the
//                  larger root hooked under the smaller (ECL-CC), so a component's root is its smallest rank
//   k_cl_flatten   parent[r] = root, roots counted, per-rank counts and report slots cleared
//   k_cl_count     one thread per pose: its root (stored over its bin), warp-aggregated integer counts per root
//   k_cl_select    one CTA: the K roots of largest (count, -rank), in that order, mapped to report slots
//   k_cl_moments<1> + k_cl_fold<1>   sums of x, y, sin, cos per reported cluster and overall: per tile of CL_TILE
//                  poses, then the tiles in order (fixed order: bitwise reproducible), the means
//   k_cl_moments<2> + k_cl_fold<2>   the centred second moments the same way; the last CTA writes the host's record
#include "kernels_common.cuh"

#include <algorithm>

namespace slamrs {

constexpr uint32_t CL_NONE = 0xffffffffu;   // excluded pose (bins stay below 2^28)
constexpr uint32_t CL_SCAN = 1024;          // words per tile of the ordered compaction (one per thread)
constexpr uint32_t CL_WARPS = 8;            // moments: warps per CTA
constexpr uint32_t CL_BATCHES = 16;         // moments: batches of 32 poses per warp
constexpr uint32_t CL_TILE = CL_WARPS * CL_BATCHES * 32u;   // poses per moment tile
constexpr uint32_t CL_SLOTS = CLUSTER_MAX_K + 1;            // reported clusters + overall
constexpr uint32_t CL_NV = 4;               // values per slot: pass 1 x, y, sin, cos; pass 2 xx, xy, yy

struct ClusterHeader {
    uint32_t n_excluded, n_clusters, n_bins, n_sel;
    uint32_t sel[CLUSTER_MAX_K];   // the reported roots (ranks), in report order
};

struct ClusterBufs {
    ClusterHeader* hdr;   // followed by the bitmap (both cleared before every call)
    uint32_t* bits;       // words
    uint32_t* wpre;       // words: occupied bins in front of each word
    uint32_t* tiles;      // ceil(words / CL_SCAN): per-tile counts, then offsets
    uint32_t* occ;        // ranks: bin id of each occupied bin
    uint32_t* parent;     // ranks
    uint32_t* counts;     // ranks: poses per root
    uint8_t* cslot;       // ranks: report slot of a root, 0xff = not reported
    uint32_t* pose_root;  // capacity: bin, then root, of each pose (CL_NONE: excluded)
    double* partials;     // ceil(capacity / CL_TILE) tiles x CL_SLOTS x CL_NV
    double* means;        // CL_SLOTS x CL_NV: mean x, mean y, S, C
    size_t words, ranks, bytes;
};

static size_t align256(size_t v) { return (v + 255u) & ~(size_t)255u; }

static ClusterBufs cluster_layout(void* base, uint32_t capacity, uint64_t bin_space) {
    ClusterBufs b{};
    b.words = (size_t)((bin_space + 31u) / 32u);
    b.ranks = (size_t)std::min<uint64_t>(capacity, bin_space);
    const size_t tiles = (b.words + CL_SCAN - 1) / CL_SCAN, mtiles = ((size_t)capacity + CL_TILE - 1) / CL_TILE;
    char* p = (char*)base;
    size_t off = 0;
    auto take = [&](size_t bytes) { char* q = p + off; off = align256(off + bytes); return q; };
    b.hdr = (ClusterHeader*)take(sizeof(ClusterHeader) + sizeof(uint32_t) * b.words);
    b.bits = (uint32_t*)(b.hdr + 1);
    b.wpre = (uint32_t*)take(sizeof(uint32_t) * b.words);
    b.tiles = (uint32_t*)take(sizeof(uint32_t) * tiles);
    b.occ = (uint32_t*)take(sizeof(uint32_t) * b.ranks);
    b.parent = (uint32_t*)take(sizeof(uint32_t) * b.ranks);
    b.counts = (uint32_t*)take(sizeof(uint32_t) * b.ranks);
    b.cslot = (uint8_t*)take(b.ranks);
    b.pose_root = (uint32_t*)take(sizeof(uint32_t) * capacity);
    b.partials = (double*)take(sizeof(double) * mtiles * CL_SLOTS * CL_NV);
    b.means = (double*)take(sizeof(double) * CL_SLOTS * CL_NV);
    b.bytes = off;
    return b;
}

size_t cluster_scratch_bytes(uint32_t capacity, uint64_t bin_space) { return cluster_layout(nullptr, capacity, bin_space).bytes; }

__device__ __forceinline__ uint32_t cl_rank(const uint32_t* __restrict__ bits, const uint32_t* __restrict__ wpre, uint32_t b) {
    return wpre[b >> 5] + (uint32_t)__popc(bits[b >> 5] & ((1u << (b & 31u)) - 1u));
}
__device__ __forceinline__ bool cl_occupied(const uint32_t* __restrict__ bits, uint32_t b) {
    return (bits[b >> 5] >> (b & 31u)) & 1u;
}

// ---------------------------------------------------------------------------------------------------- bins
__global__ void __launch_bounds__(256)
k_cl_mark(const float* __restrict__ pose, uint32_t n, MapGeom geom, KldParams kp, uint32_t* __restrict__ pose_bin,
          uint32_t* bits, ClusterHeader* hdr) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t b = CL_NONE;
    if (i < n) {
        const float x = pose[3 * (size_t)i], y = pose[3 * (size_t)i + 1], t = pose[3 * (size_t)i + 2];
        if (isfinite(x) && isfinite(y) && isfinite(t)) {
            b = kld_bin(x, y, t, geom, kp);
            if (b == kp.nbx * kp.nby * kp.theta_bins) b = CL_NONE;   // off the grid
        }
        pose_bin[i] = b;
    }
    // as k_loc_kld: one lane per distinct bin of the warp touches the bitmap, and only if the bit is not yet set
    const unsigned peers = __match_any_sync(0xffffffffu, b);
    if (b != CL_NONE && (threadIdx.x & 31u) == (unsigned)(__ffs(peers) - 1)) {
        const uint32_t bit = 1u << (b & 31u);
        uint32_t* w = &bits[b >> 5];
        if ((*(volatile const uint32_t*)w & bit) == 0u) atomicOr(w, bit);
    }
    const unsigned ex = __ballot_sync(0xffffffffu, i < n && b == CL_NONE);
    if ((threadIdx.x & 31u) == 0 && ex) atomicAdd(&hdr->n_excluded, (uint32_t)__popc(ex));
    pdl_launch_dependents();
}

// occupied bins per tile of CL_SCAN words
__global__ void __launch_bounds__(CL_SCAN) k_cl_words(const uint32_t* __restrict__ bits, uint32_t n_words,
                                                      uint32_t* __restrict__ tiles) {
    __shared__ uint32_t s_tot[33];
    pdl_wait();
    const uint32_t w = blockIdx.x * CL_SCAN + threadIdx.x;
    uint32_t total;
    block_excl_scan_u32(w < n_words ? (uint32_t)__popc(bits[w]) : 0u, s_tot, &total);
    if (threadIdx.x == 0) tiles[blockIdx.x] = total;
}

// after the tile offsets: the rank prefix of every word, the occupied bins by rank, parent[r] = r, n_bins
__global__ void __launch_bounds__(CL_SCAN)
k_cl_rank(const uint32_t* __restrict__ bits, uint32_t n_words, const uint32_t* __restrict__ tiles, uint32_t* __restrict__ wpre,
          uint32_t* __restrict__ occ, uint32_t* __restrict__ parent, ClusterHeader* hdr) {
    __shared__ uint32_t s_tot[33];
    pdl_wait();
    const uint32_t w = blockIdx.x * CL_SCAN + threadIdx.x;
    uint32_t word = w < n_words ? bits[w] : 0u;
    uint32_t total;
    uint32_t r = tiles[blockIdx.x] + block_excl_scan_u32((uint32_t)__popc(word), s_tot, &total);
    if (w < n_words) wpre[w] = r;
    if (w == n_words - 1u) hdr->n_bins = r + (uint32_t)__popc(word);
    for (; word; word &= word - 1u, ++r) {
        occ[r] = (w << 5) + (uint32_t)(__ffs(word) - 1);
        parent[r] = r;
    }
    pdl_launch_dependents();
}

// ---------------------------------------------------------------------------------------------------- components
// parent[r] <= r always holds (a root is only ever hooked under a smaller one), so the walk ends where parent[r] == r;
// each hop also points the node it left at its grandparent (intermediate pointer jumping, ECL-CC)
__device__ __forceinline__ uint32_t cl_find(uint32_t* parent, uint32_t x) {
    volatile uint32_t* p = parent;
    uint32_t cur = p[x];
    if (cur != x) {
        uint32_t prev = x, next;
        while (cur > (next = p[cur])) {
            p[prev] = next;
            prev = cur;
            cur = next;
        }
    }
    return cur;
}

__global__ void __launch_bounds__(256)
k_cl_union(const uint32_t* __restrict__ bits, const uint32_t* __restrict__ wpre, const uint32_t* __restrict__ occ,
           uint32_t* parent, const ClusterHeader* hdr, KldParams kp) {
    pdl_wait();
    const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= hdr->n_bins) return;
    const uint32_t b = occ[r], tb = kp.theta_bins;
    const uint32_t h = b % tb, cell = b / tb, bx = cell % kp.nbx, by = cell / kp.nbx;
    for (int dy = -1; dy <= 1; ++dy) {
        const int y2 = (int)by + dy;
        if (y2 < 0 || y2 >= (int)kp.nby) continue;
        for (int dx = -1; dx <= 1; ++dx) {
            const int x2 = (int)bx + dx;
            if (x2 < 0 || x2 >= (int)kp.nbx) continue;
            for (int dh = -1; dh <= 1; ++dh) {
                const uint32_t h2 = (uint32_t)((int)(h + tb) + dh) % tb;   // heading bins wrap
                const uint32_t nb = ((uint32_t)y2 * kp.nbx + (uint32_t)x2) * tb + h2;
                // every adjacent pair is joined from its smaller bin (the same bin again: theta_bins <= 2)
                if (nb <= b || !cl_occupied(bits, nb)) continue;
                uint32_t a = cl_find(parent, r), o = cl_find(parent, cl_rank(bits, wpre, nb));
                while (a != o) {   // hook the larger root under the smaller; a failed CAS retries from its new parent
                    if (a < o) {
                        const uint32_t ret = atomicCAS(&parent[o], o, a);
                        if (ret == o) break;
                        o = ret;
                    } else {
                        const uint32_t ret = atomicCAS(&parent[a], a, o);
                        if (ret == a) break;
                        a = ret;
                    }
                }
            }
        }
    }
}

__global__ void __launch_bounds__(256)
k_cl_flatten(uint32_t* parent, uint32_t* __restrict__ counts, uint8_t* __restrict__ cslot, ClusterHeader* hdr) {
    pdl_wait();
    const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
    const bool in = r < hdr->n_bins;
    bool root = false;
    if (in) {
        uint32_t x = r;
        while (parent[x] != x) x = parent[x];
        parent[r] = x;   // (another thread's walk may read it: x is an ancestor of r either way)
        root = x == r;
        counts[r] = 0u;
        cslot[r] = 0xffu;
    }
    const unsigned m = __ballot_sync(0xffffffffu, root);
    if ((threadIdx.x & 31u) == 0 && m) atomicAdd(&hdr->n_clusters, (uint32_t)__popc(m));
    pdl_launch_dependents();
}

__global__ void __launch_bounds__(256)
k_cl_count(uint32_t* __restrict__ pose_root, uint32_t n, const uint32_t* __restrict__ bits, const uint32_t* __restrict__ wpre,
           const uint32_t* __restrict__ parent, uint32_t* counts) {
    pdl_wait();
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t root = CL_NONE;
    if (i < n) {
        const uint32_t b = pose_root[i];
        if (b != CL_NONE) root = parent[cl_rank(bits, wpre, b)];
        pose_root[i] = root;
    }
    const unsigned peers = __match_any_sync(0xffffffffu, root);
    if (root != CL_NONE && (threadIdx.x & 31u) == (unsigned)(__ffs(peers) - 1)) atomicAdd(&counts[root], (uint32_t)__popc(peers));
    pdl_launch_dependents();
}

// One CTA, K rounds: round j takes the largest key below round j - 1's over the roots, key = count << 32 | ~rank
// (count descending, then rank -- hence label -- ascending; keys are distinct)
constexpr uint32_t CL_SELECT = 1024;
__global__ void __launch_bounds__(CL_SELECT)
k_cl_select(const uint32_t* __restrict__ parent, const uint32_t* __restrict__ counts, uint8_t* __restrict__ cslot,
            ClusterHeader* hdr, uint32_t k) {
    __shared__ unsigned long long s_best[CL_SELECT / 32];
    pdl_wait();
    const uint32_t n_bins = hdr->n_bins;
    const uint32_t lane = threadIdx.x & 31u, wid = threadIdx.x >> 5;
    unsigned long long prev = ~0ull;
    uint32_t j = 0;
    for (; j < k; ++j) {
        unsigned long long best = 0ull;
        for (uint32_t r = threadIdx.x; r < n_bins; r += CL_SELECT) {
            if (parent[r] != r) continue;
            const unsigned long long key = ((unsigned long long)counts[r] << 32) | (unsigned long long)(~r);
            if (key < prev && key > best) best = key;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) best = max(best, __shfl_xor_sync(0xffffffffu, best, o));
        if (lane == 0) s_best[wid] = best;
        __syncthreads();
        best = s_best[lane];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) best = max(best, __shfl_xor_sync(0xffffffffu, best, o));
        __syncthreads();   // (s_best is reused by the next round)
        if (best == 0ull) break;   // (block-uniform) every root is taken
        if (threadIdx.x == 0) {
            const uint32_t root = ~(uint32_t)best;
            hdr->sel[j] = root;
            cslot[root] = (uint8_t)j;
        }
        prev = best;
    }
    if (threadIdx.x == 0) hdr->n_sel = j;
    pdl_launch_dependents();
}

// ---------------------------------------------------------------------------------------------------- moments
// A warp takes batches of 32 consecutive poses. For the overall set and then for each reported slot present in the
// batch it folds the lanes' values with the xor butterfly (lanes outside the set add 0), and lane 0 adds the result to
// the warp's accumulators in shared memory: the order of every addition is fixed by the pose indices alone. The CTA then
// adds its warps' accumulators in warp order into its tile's partials.
template <int PASS>
__device__ __forceinline__ void cl_values(float x, float y, float t, const double* m, double v[CL_NV]) {
    if (PASS == 1) {
        double s, c;
        sincos((double)t, &s, &c);
        v[0] = (double)x; v[1] = (double)y; v[2] = s; v[3] = c;
    } else {
        const double dx = __dsub_rn((double)x, m[0]), dy = __dsub_rn((double)y, m[1]);
        v[0] = __dmul_rn(dx, dx); v[1] = __dmul_rn(dx, dy); v[2] = __dmul_rn(dy, dy); v[3] = 0.0;
    }
}

__device__ __forceinline__ void cl_warp_add(double v[CL_NV], bool in, double* acc) {
    double s[CL_NV];
#pragma unroll
    for (int c = 0; c < (int)CL_NV; ++c) {
        s[c] = in ? v[c] : 0.0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s[c] = __dadd_rn(s[c], __shfl_xor_sync(0xffffffffu, s[c], o));
    }
    if ((threadIdx.x & 31u) == 0) {
#pragma unroll
        for (int c = 0; c < (int)CL_NV; ++c) acc[c] = __dadd_rn(acc[c], s[c]);
    }
}

template <int PASS>
__global__ void __launch_bounds__(CL_WARPS * 32)
k_cl_moments(const float* __restrict__ pose, uint32_t n, const uint32_t* __restrict__ pose_root,
             const uint8_t* __restrict__ cslot, const double* __restrict__ means, double* __restrict__ partials, uint32_t k) {
    __shared__ double s_acc[CL_WARPS][CL_SLOTS][CL_NV];
    const uint32_t lane = threadIdx.x & 31u, wid = threadIdx.x >> 5;
    for (uint32_t e = threadIdx.x; e < CL_WARPS * CL_SLOTS * CL_NV; e += blockDim.x) (&s_acc[0][0][0])[e] = 0.0;
    __syncthreads();
    pdl_wait();
    const uint32_t base = blockIdx.x * CL_TILE;
    for (uint32_t it = 0; it < CL_BATCHES; ++it) {
        const uint32_t i = base + (it * CL_WARPS + wid) * 32u + lane;
        bool valid = false;
        uint32_t s = 0xffu;
        float x = 0.0f, y = 0.0f, t = 0.0f;
        if (i < n) {
            const uint32_t root = pose_root[i];
            valid = root != CL_NONE;
            if (valid) {
                s = cslot[root];
                x = pose[3 * (size_t)i]; y = pose[3 * (size_t)i + 1]; t = pose[3 * (size_t)i + 2];
            }
        }
        if (!__any_sync(0xffffffffu, valid)) continue;
        double v[CL_NV];
        cl_values<PASS>(x, y, t, means + (size_t)k * CL_NV, v);
        cl_warp_add(v, valid, s_acc[wid][k]);   // overall
        unsigned pending = __ballot_sync(0xffffffffu, valid && s < k);
        while (pending) {   // (warp-uniform)
            const uint32_t s0 = __shfl_sync(0xffffffffu, s, __ffs(pending) - 1);
            const bool in = valid && s == s0;
            if (PASS == 2) cl_values<PASS>(x, y, t, means + (size_t)s0 * CL_NV, v);
            cl_warp_add(v, in, s_acc[wid][s0]);
            pending &= ~__ballot_sync(0xffffffffu, in);
        }
    }
    __syncthreads();
    for (uint32_t e = threadIdx.x; e < CL_SLOTS * CL_NV; e += blockDim.x) {
        double sum = 0.0;
        for (uint32_t w = 0; w < CL_WARPS; ++w) sum = __dadd_rn(sum, (&s_acc[w][0][0])[e]);
        partials[(size_t)blockIdx.x * CL_SLOTS * CL_NV + e] = sum;
    }
    pdl_launch_dependents();
}

// One CTA: the tiles' partials in tile order, then pass 1 the means (means[s] = {mean x, mean y, S, C}), pass 2 the
// record in page-locked host memory
template <int PASS>
__global__ void __launch_bounds__(CL_SLOTS * CL_NV)
k_cl_fold(const double* __restrict__ partials, uint32_t n_tiles, uint32_t n, uint32_t k, const ClusterHeader* hdr,
          const uint32_t* __restrict__ occ, const uint32_t* __restrict__ counts, double* means, ClusterOutput* host_out) {
    __shared__ double s_sum[CL_SLOTS * CL_NV];
    pdl_wait();
    const uint32_t e = threadIdx.x;
    double sum = 0.0;
    for (uint32_t t = 0; t < n_tiles; ++t) sum = __dadd_rn(sum, partials[(size_t)t * CL_SLOTS * CL_NV + e]);
    s_sum[e] = sum;
    __syncthreads();
    const uint32_t n_sel = hdr->n_sel;
    const uint32_t s = e;   // thread s < CL_SLOTS finishes slot s (slot k: overall)
    if (s > k || (s < k && s >= n_sel)) {
        if (PASS == 2 && s < k) memset(&host_out->clusters[s], 0, sizeof(slamrs_gpu_pose_cluster));
        return;
    }
    const uint32_t count = s == k ? n - hdr->n_excluded : counts[hdr->sel[s]];
    const double* q = s_sum + (size_t)s * CL_NV;
    if (PASS == 1) {
        double* m = means + (size_t)s * CL_NV;
        const double c = (double)count;
        m[0] = count ? __ddiv_rn(q[0], c) : 0.0;
        m[1] = count ? __ddiv_rn(q[1], c) : 0.0;
        m[2] = q[2];
        m[3] = q[3];
        return;
    }
    slamrs_gpu_pose_cluster out;
    memset(&out, 0, sizeof(out));
    if (count) {
        const double c = (double)count, *m = means + (size_t)s * CL_NV;
        out.count = count;
        out.label = s == k ? 0ull : occ[hdr->sel[s]];
        out.weight = __ddiv_rn(c, (double)n);
        out.mean[0] = m[0];
        out.mean[1] = m[1];
        out.mean[2] = atan2(m[2], m[3]);
        out.cov_xx = __ddiv_rn(q[0], c);
        out.cov_xy = __ddiv_rn(q[1], c);
        out.cov_yy = __ddiv_rn(q[2], c);
        const double r = __ddiv_rn(__dsqrt_rn(__dadd_rn(__dmul_rn(m[2], m[2]), __dmul_rn(m[3], m[3]))), c);
        out.var_theta = __dmul_rn(-2.0, log(r));
    }
    if (s == k) {
        host_out->stats.n_poses = n;
        host_out->stats.n_excluded = hdr->n_excluded;
        host_out->stats.n_bins = hdr->n_bins;
        host_out->stats.n_clusters = hdr->n_clusters;
        host_out->stats.overall = out;
    } else {
        host_out->clusters[s] = out;
    }
    __threadfence_system();
}

cudaError_t launch_pose_clusters(cudaStream_t stream, const float* pose, uint32_t n, uint32_t capacity, MapGeom geom,
                                 const KldParams& bins, uint32_t k, void* scratch, ClusterOutput* host_out,
                                 uint64_t* launches) {
    const uint64_t bin_space = (uint64_t)bins.nbx * bins.nby * bins.theta_bins;
    const ClusterBufs b = cluster_layout(scratch, capacity, bin_space);
    const uint32_t n_words = (uint32_t)b.words, n_tiles = (uint32_t)((b.words + CL_SCAN - 1) / CL_SCAN);
    const uint32_t max_ranks = (uint32_t)std::min<uint64_t>(n, bin_space);
    const uint32_t pose_blocks = (n + 255u) / 256u, rank_blocks = (max_ranks + 255u) / 256u;
    const uint32_t m_tiles = (n + CL_TILE - 1u) / CL_TILE;
    cudaError_t e = cudaMemsetAsync(b.hdr, 0, sizeof(ClusterHeader) + sizeof(uint32_t) * b.words, stream);
    if (e != cudaSuccess) return e;
    k_cl_mark<<<pose_blocks, 256, 0, stream>>>(pose, n, geom, bins, b.pose_root, b.bits, b.hdr);
    if ((e = launch_pdl(k_cl_words, dim3(n_tiles), dim3(CL_SCAN), 0, stream, b.bits, n_words, b.tiles)) != cudaSuccess) return e;
    launch_tile_offsets(stream, b.tiles, n_tiles);   // (plain launch: k_loc_free_scan does not wait for a predecessor)
    if ((e = launch_pdl(k_cl_rank, dim3(n_tiles), dim3(CL_SCAN), 0, stream, b.bits, n_words, b.tiles, b.wpre, b.occ, b.parent,
                        b.hdr)) != cudaSuccess) return e;
    if ((e = launch_pdl(k_cl_union, dim3(rank_blocks), dim3(256), 0, stream, b.bits, b.wpre, b.occ, b.parent, b.hdr, bins)) !=
        cudaSuccess) return e;
    if ((e = launch_pdl(k_cl_flatten, dim3(rank_blocks), dim3(256), 0, stream, b.parent, b.counts, b.cslot, b.hdr)) !=
        cudaSuccess) return e;
    if ((e = launch_pdl(k_cl_count, dim3(pose_blocks), dim3(256), 0, stream, b.pose_root, n, b.bits, b.wpre, b.parent,
                        b.counts)) != cudaSuccess) return e;
    if ((e = launch_pdl(k_cl_select, dim3(1), dim3(CL_SELECT), 0, stream, b.parent, b.counts, b.cslot, b.hdr, k)) != cudaSuccess)
        return e;
    if ((e = launch_pdl(k_cl_moments<1>, dim3(m_tiles), dim3(CL_WARPS * 32), 0, stream, pose, n, b.pose_root, b.cslot, b.means,
                        b.partials, k)) != cudaSuccess) return e;
    if ((e = launch_pdl(k_cl_fold<1>, dim3(1), dim3(CL_SLOTS * CL_NV), 0, stream, b.partials, m_tiles, n, k, b.hdr, b.occ,
                        b.counts, b.means, host_out)) != cudaSuccess) return e;
    if ((e = launch_pdl(k_cl_moments<2>, dim3(m_tiles), dim3(CL_WARPS * 32), 0, stream, pose, n, b.pose_root, b.cslot, b.means,
                        b.partials, k)) != cudaSuccess) return e;
    if ((e = launch_pdl(k_cl_fold<2>, dim3(1), dim3(CL_SLOTS * CL_NV), 0, stream, b.partials, m_tiles, n, k, b.hdr, b.occ,
                        b.counts, b.means, host_out)) != cudaSuccess) return e;
    *launches = 12;
    return cudaGetLastError();
}

}  // namespace slamrs
