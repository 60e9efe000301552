// The grid copies of resampling (`value.clone()`, particle.rs:97-100): k_copy (whole grids),
// k_copy_prepare / k_copy_boxed / k_commit_boxes (informed extents, whole tiles). With deferred copies
// (PlanArgs::alias_of) the same kernels run on the short list of clones that are about to be written.
#include "kernels_common.cuh"

namespace slamrs {

// =============================================================================== k_copy
// Grid copies (the `value.clone()` of particle.rs:97-100). Pure streaming: 128-bit loads that
// bypass L1, four in flight per thread, then 128-bit stores. Copies of the same source are
// adjacent in the list, so one work item = 16 KiB of a source grid fanned out to up to
// COPY_FAN destinations: the source is read once per sub-run instead of once per copy, which
// makes the kernel write-bound (D grids written, D / COPY_FAN + distinct sources read).
// CTAs stride over (leader, chunk) items; list lengths are read from device memory so that no
// host round trip sits between planning and copying.

constexpr int COPY_THREADS = 256;
constexpr int COPY_UNROLL = 2;
constexpr uint32_t COPY_ITEM_V8 = COPY_THREADS * COPY_UNROLL;  // 32-byte units per work item (16 KiB)
constexpr int COPY_CTAS_PER_SM = 32;  // measured on B200: 6.37 TB/s moved at 32/SM vs 5.72 TB/s at 8/SM (tools/bw_probe.cu)


__global__ void __launch_bounds__(COPY_THREADS)
k_copy(const CopyItem* __restrict__ items, const uint32_t* __restrict__ leaders,
       const unsigned long long* __restrict__ n_items, const unsigned long long* __restrict__ n_leaders,
       uint32_t v8_per_grid) {
    const unsigned long long n = *n_items;
    const unsigned long long nl = leaders ? *n_leaders : n;
    const uint32_t chunks = (v8_per_grid + COPY_ITEM_V8 - 1) / COPY_ITEM_V8;
    const unsigned long long total = nl * chunks;
    for (unsigned long long w = blockIdx.x; w < total; w += gridDim.x) {
        const unsigned long long q = w / chunks;
        const uint32_t c = (uint32_t)(w - q * chunks);
        const unsigned long long k = leaders ? leaders[q] : q;
        const CopyItem it = items[k];
        uint32_t fan = 1;
        if (leaders) {
            while (fan < COPY_FAN && k + fan < n && items[k + fan].src == it.src) fan++;
        }
        const V8* src = reinterpret_cast<const V8*>(it.src);
        const uint32_t base = c * COPY_ITEM_V8 + threadIdx.x;
        V8 v[COPY_UNROLL];
#pragma unroll
        for (int u = 0; u < COPY_UNROLL; ++u) {
            const uint32_t i = base + u * COPY_THREADS;
            if (i < v8_per_grid) v[u] = ld_stream_v8(src + i);
        }
        for (uint32_t f = 0; f < fan; ++f) {
            V8* dst = reinterpret_cast<V8*>(items[k + f].dst);
#pragma unroll
            for (int u = 0; u < COPY_UNROLL; ++u) {
                const uint32_t i = base + u * COPY_THREADS;
                if (i < v8_per_grid) st_stream_v8(dst + i, v[u]);
            }
        }
    }
}

void launch_copy(cudaStream_t stream, const CopyItem* items, const uint32_t* leaders,
                 const unsigned long long* n_items, const unsigned long long* n_leaders, size_t cells_per_grid,
                 int num_sms) {
    const uint32_t v8 = (uint32_t)(cells_per_grid / 8);  // cells_per_grid is a multiple of 32 cells
    k_copy<<<num_sms * COPY_CTAS_PER_SM, COPY_THREADS, 0, stream>>>(items, leaders, n_items, n_leaders, v8);
}

// =============================================================================== k_copy_boxed
// Extent-limited grid copy. A grid is zero outside its informed extent, so cloning it means: copy the
// source's extent and clear whatever else the destination slot's previous tenant had informed. The
// extent is kept per band of 8 rows (slam_device.cuh): k_copy_prepare turns every fan-out sub-run into
// one CopyJob (source, destinations, their band tables, the band-aligned arc of slot rows to visit);
// k_copy_boxed takes one (job, band) item per single-warp CTA: it reads the 17 band entries, covers the
// source's columns and the destinations' old columns with one arc U of 32-byte units, rounds U outward
// to whole tiles when the slot is tiled (one instruction of the warp = one 1 KiB tile = one DRAM page),
// streams the 8 rows x U of the source (zero outside the source's range) into every destination and
// writes the destinations' new band entries. UNROLL independent 256-bit loads are in flight per lane;
// bytes that really moved are counted on the device and are what bench.py's roofline_copy uses.

// A job works in PHYSICAL slot coordinates. x: 32-byte units of one slot row, on a ring when the slot
// width is a power of two >= 256 (windowed slots wrap); y: rows on the ring of the slot's rows (ring size =
// slot height for windowed slots, unbounded otherwise). An "arc" is (start, length).
struct alignas(16) CopyJob {
    const uint32_t* src;
    const uint32_t* src_bands;
    uint32_t fan;
    uint32_t uy_start, uy_len;  // arc of slot rows to visit, both multiples of BAND_ROWS
    uint32_t pad;
    uint32_t* dst[COPY_FAN];
    uint32_t* dst_bands[COPY_FAN];
};
static_assert(sizeof(CopyJob) % 16 == 0, "CopyJob is fetched as 16-byte pieces");
constexpr int COPY_JOB_V4 = (int)(sizeof(CopyJob) / 16);
static_assert(COPY_JOB_V4 <= 32, "one warp fetches a job");

__device__ __forceinline__ bool meta_empty(const SlotMeta& m) { return m.x1 <= m.x0 || m.y1 <= m.y0; }

// smallest arc (of those starting at either operand's start) that covers arcs a and b on the ring
__device__ __forceinline__ void arc_cover(uint32_t& a_start, uint32_t& a_len, uint32_t b_start, uint32_t b_len,
                                          uint32_t mask, uint32_t ring) {
    if (b_len == 0u) return;
    if (a_len == 0u) { a_start = b_start; a_len = b_len; return; }
    // 64-bit: with an unbounded "ring" (no rotation / no window) the sums may exceed 32 bits
    const unsigned long long l1 = max((unsigned long long)a_len, (unsigned long long)((b_start - a_start) & mask) + b_len);
    const unsigned long long l2 = max((unsigned long long)b_len, (unsigned long long)((a_start - b_start) & mask) + a_len);
    if (l2 < l1) { a_start = b_start; a_len = (uint32_t)min(l2, (unsigned long long)ring); }
    else { a_len = (uint32_t)min(l1, (unsigned long long)ring); }
    if (a_len >= ring) { a_start = 0u; a_len = ring; }
}

// band-aligned arc of physical rows covered by logical rows [y0, y1)
__device__ __forceinline__ void row_arc(const MapGeom& geom, int y0, int y1, uint32_t& start, uint32_t& len) {
    const uint32_t b0 = (uint32_t)y0 / BAND_ROWS * BAND_ROWS, b1 = ((uint32_t)y1 + BAND_ROWS - 1u) / BAND_ROWS * BAND_ROWS;
    start = b0 & geom.ymask;
    len = b1 - b0;
}

// Waits until the owner of a source slot has published `wait_epoch` in its SlotMeta (pulls without a barrier across
// the GPUs: the owner's ray update stores it once the slot is complete -- cells, band entries, box). Bounded like the
// step barrier; a handle that has given up does not wait again. Called by one lane; the caller re-converges.
__device__ __forceinline__ void wait_source_epoch(const SlotMeta* src_meta, uint32_t wait_epoch, unsigned long long timeout_ns,
                                                  StepCounters* counters) {
    if (*reinterpret_cast<volatile unsigned long long*>(&counters->barrier_timeout) != 0ull) return;
    unsigned long long t0, now;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    for (;;) {
        uint32_t seen;
        asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(seen) : "l"(&src_meta->pad0) : "memory");
        if (seen == wait_epoch) break;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
        if (now - t0 > timeout_ns) { counters->barrier_timeout = 1ull; break; }
        __nanosleep(200);
    }
}

// One warp turns the fan-out sub-run q of the copy list into a CopyJob (*job: global or shared memory).
__device__ __forceinline__ void prepare_job(const CopyItem* __restrict__ items, const uint32_t* __restrict__ leaders,
                                            unsigned long long n, unsigned long long q, CopyJob* job, const MapGeom& geom,
                                            StepCounters* counters, uint32_t wait_epoch, unsigned long long timeout_ns,
                                            const SlotMeta* meta_base = nullptr, const uint32_t* readers = nullptr,
                                            const uint32_t* done = nullptr) {
    const int lane = threadIdx.x & 31;
    const uint32_t ymask = geom.ymask, yring = geom.ymask == 0xffffffffu ? 0xffffffffu : geom.ph;
    const unsigned long long k = leaders ? leaders[q] : q;
    const bool have = lane < (int)COPY_FAN && k + lane < n && (leaders != nullptr || lane == 0);
    CopyItem it{};
    if (have) it = items[k + lane];
    const unsigned long long src0 = __shfl_sync(0xffffffffu, (unsigned long long)(uintptr_t)it.src, 0);
    const unsigned same = __ballot_sync(0xffffffffu, have && (unsigned long long)(uintptr_t)it.src == src0);
    const uint32_t fan = (uint32_t)(__ffs(~same) - 1);   // leading run of items that share the source
    SlotMeta sm{0, 0, 0, 0, 0, 0, 0, 0}, dm{0, 0, 0, 0, 0, 0, 0, 0};
    if (wait_epoch != 0u) {
        if (lane == 0) wait_source_epoch(it.src_meta, wait_epoch, timeout_ns, counters);
        // A destination is a slot no survivor owns -- but the cells it still holds may be the ROOT that surviving clones
        // of a dropped particle read in this very ray update (they become private there). The pull runs concurrently
        // with that kernel, so it waits until every such reader is done with the slot (the owners' own protocol:
        // readers[] = clone halves listed for the slot, done[] = those that have finished).
#ifndef SLAMRS_TEST_NO_READER_WAIT   /* (a build without this wait must fail tests/test_gpu_multi.py::test_sharded_state_at_scale...) */
        if (readers != nullptr && lane < (int)fan) {
            const size_t slot = (size_t)(it.dst_meta - meta_base);
            const uint32_t want = readers[slot];
            if (want != 0u && *reinterpret_cast<volatile unsigned long long*>(&counters->barrier_timeout) == 0ull) {
                unsigned long long t0, now;
                asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
                for (;;) {
                    uint32_t seen;
                    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(done + slot) : "memory");
                    if (seen >= want) break;
                    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
                    if (now - t0 > timeout_ns) { counters->barrier_timeout = 1ull; break; }
                    __nanosleep(200);
                }
            }
        }
#endif
        __syncwarp();
        __threadfence_system();
    }
    if (lane == 0) {   // (not through L1: a peer has just written it)
        const int4 box = __ldcv(reinterpret_cast<const int4*>(it.src_meta));
        sm.x0 = box.x; sm.y0 = box.y; sm.x1 = box.z; sm.y1 = box.w;
    }
    if (lane < (int)fan) dm = *it.dst_meta;
    // rows: the destinations' old rows (to clear) and the source's rows, as band-aligned arcs
    uint32_t oy_start = 0u, oy_len = 0u;
    if (lane < (int)fan && !meta_empty(dm)) row_arc(geom, dm.y0, dm.y1, oy_start, oy_len);
    uint32_t uy_start = 0u, uy_len = 0u;
    if (lane == 0 && !meta_empty(sm)) row_arc(geom, sm.y0, sm.y1, uy_start, uy_len);
    for (uint32_t f = 0; f < fan; ++f) {
        const uint32_t bys = __shfl_sync(0xffffffffu, oy_start, (int)f), byl = __shfl_sync(0xffffffffu, oy_len, (int)f);
        if (lane == 0) arc_cover(uy_start, uy_len, bys, byl, ymask, yring);
    }
    if (lane < (int)COPY_FAN) {
        job->dst[lane] = lane < (int)fan ? it.dst : nullptr;
        job->dst_bands[lane] = lane < (int)fan ? it.dst_bands : nullptr;
    }
    if (lane == 0) {
        job->src = it.src; job->src_bands = it.src_bands; job->fan = fan;
        job->uy_start = uy_start; job->uy_len = uy_len;
        job->pad = 0u;
        if (uy_len) atomicMax(&counters->copy_max_rows, (unsigned long long)uy_len);
    }
}

// one warp per job
__global__ void __launch_bounds__(256)
k_copy_prepare(const CopyItem* __restrict__ items, const uint32_t* __restrict__ leaders,
               const unsigned long long* __restrict__ n_items, const unsigned long long* __restrict__ n_leaders,
               CopyJob* __restrict__ jobs, MapGeom geom, StepCounters* counters, uint32_t wait_epoch,
               unsigned long long timeout_ns) {
    const unsigned long long n = *n_items;
    const unsigned long long nl = leaders ? *n_leaders : n;
    const unsigned long long q = (unsigned long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (q >= nl) return;
    prepare_job(items, leaders, n, q, jobs + q, geom, counters, wait_epoch, timeout_ns);
}

// CTAs are single warps: a band is a few hundred 32-byte elements, and with more warps per CTA the
// barriers per item dominate (profiles/r1_copy_tuning.md).
constexpr int BOX_THREADS = 32;
#ifndef BOX_CTAS
#define BOX_CTAS 256
#endif
#ifndef BOX_UNROLL
#define BOX_UNROLL 8   // loads in flight per lane: 8 x 12 resident warps measured 2.5 % above 4 x 24 (same bytes in flight,
#define BOX_MINB 12    // half the dependent round trips per item)
#endif
constexpr int BOX_CTAS_PER_SM = BOX_CTAS;
#ifndef BOX_SHORT_CTAS
#define BOX_SHORT_CTAS 48   // CTAs per SM for a short list (a few hundred jobs)
#endif

// One band (BAND_ROWS slot rows) of one job, by one warp: the source's columns of the band into every destination, the
// rest of what the destinations had informed there cleared, the destinations' band entries rewritten.
template <int UNROLL>
__device__ __forceinline__ void copy_job_band(const CopyJob& s_job, uint32_t bi, const MapGeom& geom, uint32_t& moved,
                                              const uint32_t* src_entries = nullptr /* [bi]: the source's band entries, prefetched */) {
    const int lane = threadIdx.x & 31;
    const uint32_t row_units = geom.pw / 8u;
    const bool tiled = geom.tiled != 0u;
    constexpr uint32_t TILE_UNITS = TILE_COLS / 8u;   // 32-byte units per tile row
    const uint32_t umask = geom.xmask == 0xffffffffu ? 0xffffffffu : (geom.xmask >> 3);
    const uint32_t uring = geom.xmask == 0xffffffffu ? 0xffffffffu : row_units;
    if (bi * BAND_ROWS >= s_job.uy_len) return;
    const uint32_t prow0 = (s_job.uy_start + bi * BAND_ROWS) & geom.ymask;   // first slot row of the band
    const uint32_t pb = prow0 / BAND_ROWS;
    const uint32_t fan = s_job.fan;
    // ---- the 17 band entries: lane f < fan = destination f's old columns, lane 31 = the source's
    uint32_t a_start = 0u, a_len = 0u;      // this lane's arc in destination units
    uint32_t src_entry = 0u;
    if ((uint32_t)lane < fan) {
        const uint32_t e = s_job.dst_bands[lane][pb];
        if (e) {
            a_start = (phys_col(geom, e & 0xffffu) >> 3) & umask;
            a_len = ((e >> 16) - (e & 0xffffu)) >> 3;
        }
    } else if (lane == 31) {
        src_entry = src_entries ? src_entries[bi] : __ldg(&s_job.src_bands[pb]);
    }
    src_entry = __shfl_sync(0xffffffffu, src_entry, 31);
    uint32_t n_start = 0u, n_len = 0u;   // the source's columns (same place in source and destination)
    if (src_entry) {
        const uint32_t sx0 = src_entry & 0xffffu;
        n_len = ((src_entry >> 16) - sx0) >> 3;
        n_start = (phys_col(geom, sx0) >> 3) & umask;
        if (lane == 31) { a_start = n_start; a_len = n_len; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {   // cover of all arcs, reduced to lane 0
        const uint32_t bs = __shfl_down_sync(0xffffffffu, a_start, o), bl = __shfl_down_sync(0xffffffffu, a_len, o);
        arc_cover(a_start, a_len, bs, bl, umask, uring);
    }
    uint32_t u_start = __shfl_sync(0xffffffffu, a_start, 0), uw = __shfl_sync(0xffffffffu, a_len, 0);
    if (tiled && uw != 0u) {   // whole tiles: every DRAM page the band touches is written in full
        uw = ((u_start & (TILE_UNITS - 1u)) + uw + TILE_UNITS - 1u) & ~(TILE_UNITS - 1u);
        u_start &= ~(TILE_UNITS - 1u);
        if (uw >= uring) { u_start = 0u; uw = uring; }
    }
    if (uw != 0u) {
        const uint32_t count = BAND_ROWS * uw;
        const V8* src = reinterpret_cast<const V8*>(s_job.src);
        for (uint32_t base = lane; base < count; base += BOX_THREADS * UNROLL) {
            V8 v[UNROLL];
            uint32_t off[UNROLL];   // unit offset inside a destination slot (< 2^28)
#pragma unroll
            for (int u = 0; u < UNROLL; ++u) {
                const uint32_t i = base + u * BOX_THREADS;
                off[u] = 0xffffffffu;
                v[u].a = make_uint4(0u, 0u, 0u, 0u); v[u].b = v[u].a;
                if (i < count) {
                    // row-major slots: a lane walks the band's rows; tiled slots: 32 lanes = one tile (1 KiB)
                    const uint32_t rr = tiled ? (i / TILE_UNITS) % BAND_ROWS : i / uw;
                    const uint32_t cu = tiled ? i / (TILE_UNITS * BAND_ROWS) * TILE_UNITS + i % TILE_UNITS : i - rr * uw;
                    const uint32_t py = prow0 + rr;                  // same slot row in source and destination
                    const uint32_t du = (u_start + cu) & umask;      // destination unit on the ring
                    off[u] = phys_unit(geom, py, du);
                    if (((du - n_start) & umask) < n_len) {
                        v[u] = ld_stream_v8(src + off[u]);
                        moved++;
                    }
                }
            }
            for (uint32_t f = 0; f < fan; ++f) {
                V8* dst = reinterpret_cast<V8*>(s_job.dst[f]);
#pragma unroll
                for (int u = 0; u < UNROLL; ++u)
                    if (off[u] != 0xffffffffu) { st_stream_v8(dst + off[u], v[u]); moved++; }
            }
        }
    }
    // the destinations now hold the source's columns in this band (or nothing)
    if ((uint32_t)lane < fan) s_job.dst_bands[lane][pb] = src_entry;
}

template <int UNROLL, int MINB>
__global__ void __launch_bounds__(BOX_THREADS, MINB)
k_copy_boxed(const CopyJob* __restrict__ jobs, const unsigned long long* __restrict__ n_jobs, MapGeom geom,
             StepCounters* counters) {
    __shared__ CopyJob s_job;
    const unsigned long long nl = *n_jobs;
    if (nl == 0) return;
    const int lane = threadIdx.x;
    const uint32_t bands = max(1u, (uint32_t)counters->copy_max_rows / BAND_ROWS);   // work items per job
    const uint32_t total = (uint32_t)min(nl * bands, 0xffffffffull);
    uint32_t moved = 0;   // 32-byte units read + written by this lane
    uint4 next_job = make_uint4(0u, 0u, 0u, 0u);
    if (lane < COPY_JOB_V4 && blockIdx.x < total)
        next_job = reinterpret_cast<const uint4*>(jobs + blockIdx.x / bands)[lane];
    for (uint32_t w = blockIdx.x; w < total; w += gridDim.x) {
        const uint32_t q = w / bands;
        const uint32_t bi = w - q * bands;
        __syncwarp();   // the previous item's job is no longer read
        if (lane < COPY_JOB_V4) {
            reinterpret_cast<uint4*>(&s_job)[lane] = next_job;
            const unsigned long long wn = (unsigned long long)w + gridDim.x;
            if (wn < total) next_job = reinterpret_cast<const uint4*>(jobs + (uint32_t)wn / bands)[lane];
        }
        __syncwarp();
        copy_job_band<UNROLL>(s_job, bi, geom, moved);
    }
    // bytes actually moved, for the roofline: one atomic per warp = per CTA
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) moved += __shfl_down_sync(0xffffffffu, moved, o);
    if (lane == 0 && moved) atomicAdd(&counters->copy_bytes, (unsigned long long)moved * 32ull);
}

// =============================================================================== k_pull
// Pulls of remote sources without a barrier across the GPUs (world > 1, default path): one CTA per job. Warp 0 waits
// until the source's owner has published this step's epoch in the slot's SlotMeta (its ray update has left the slot
// complete), builds the job in shared memory, and the CTA's warps copy its bands over NVLink. Runs on the side stream
// behind the planner, concurrently with this GPU's own ray update: a pull starts as soon as ITS source is ready.
constexpr int PULL_THREADS = 256;
constexpr uint32_t PULL_SPLIT = 4;          // CTAs per job: a pull is bound by NVLink round trips, not by bytes
constexpr uint32_t PULL_MAX_BANDS = 512;    // band entries of the source prefetched per job (more: read one by one)
__global__ void __launch_bounds__(PULL_THREADS)
k_pull(const CopyItem* __restrict__ items, const uint32_t* __restrict__ leaders, const unsigned long long* __restrict__ n_items,
       const unsigned long long* __restrict__ n_leaders, MapGeom geom, StepCounters* counters, uint32_t wait_epoch,
       unsigned long long timeout_ns, const SlotMeta* __restrict__ meta_base, const uint32_t* __restrict__ readers,
       const uint32_t* __restrict__ done) {
    __shared__ CopyJob s_job;
    __shared__ uint32_t s_src_entries[PULL_MAX_BANDS];
    const unsigned long long n = *n_items;
    const unsigned long long nl = leaders ? *n_leaders : n;
    const uint32_t warp = threadIdx.x >> 5, n_warps = blockDim.x >> 5;
    uint32_t moved = 0;
    for (unsigned long long w = blockIdx.x; w < nl * PULL_SPLIT; w += gridDim.x) {
        const unsigned long long q = w / PULL_SPLIT;
        const uint32_t part = (uint32_t)(w - q * PULL_SPLIT);
        __syncthreads();   // the previous job is no longer read
        if (warp == 0) prepare_job(items, leaders, n, q, &s_job, geom, counters, wait_epoch, timeout_ns, meta_base, readers, done);
        __syncthreads();
        const uint32_t bands = s_job.uy_len / BAND_ROWS;
        // the source's band entries of this CTA's bands in one round trip
        const bool prefetched = bands <= PULL_MAX_BANDS;
        if (prefetched) {
            for (uint32_t bi = part * n_warps + threadIdx.x / 32u + (threadIdx.x & 31u) * PULL_SPLIT * n_warps; bi < bands;
                 bi += 32u * PULL_SPLIT * n_warps) {
                const uint32_t prow0 = (s_job.uy_start + bi * BAND_ROWS) & geom.ymask;
                s_src_entries[bi] = __ldcv(&s_job.src_bands[prow0 / BAND_ROWS]);
            }
            __syncthreads();
        }
        for (uint32_t bi = part * n_warps + warp; bi < bands; bi += PULL_SPLIT * n_warps)
            copy_job_band<4>(s_job, bi, geom, moved, prefetched ? s_src_entries : nullptr);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) moved += __shfl_down_sync(0xffffffffu, moved, o);
    if ((threadIdx.x & 31) == 0 && moved) atomicAdd(&counters->copy_bytes, (unsigned long long)moved * 32ull);
}
void launch_pull(cudaStream_t stream, const CopyItem* items, const uint32_t* leaders, const unsigned long long* n_items,
                 const unsigned long long* n_leaders, uint32_t max_items, MapGeom geom, StepCounters* counters, int num_sms,
                 uint32_t wait_epoch, unsigned long long timeout_ns, const SlotMeta* meta_base, const uint32_t* readers,
                 const uint32_t* done) {
    const unsigned long long want = (unsigned long long)(max_items ? max_items : 1u) * PULL_SPLIT;
    const uint32_t grid = (uint32_t)(want < 2ull * (unsigned long long)num_sms ? want : 2ull * (unsigned long long)num_sms);
    k_pull<<<grid, PULL_THREADS, 0, stream>>>(items, leaders, n_items, n_leaders, geom, counters, wait_epoch, timeout_ns, meta_base,
                                              readers, done);
}

void launch_copy_boxed(cudaStream_t stream, const CopyItem* items, const uint32_t* leaders,
                       const unsigned long long* n_items, const unsigned long long* n_leaders, uint32_t max_items,
                       void* jobs, MapGeom geom, StepCounters* counters, int num_sms, bool short_list, uint32_t wait_epoch,
                       unsigned long long timeout_ns) {
    const uint32_t blocks = (max_items + 7u) / 8u;
    k_copy_prepare<<<blocks ? blocks : 1, 256, 0, stream>>>(items, leaders, n_items, n_leaders, (CopyJob*)jobs, geom, counters,
                                                            wait_epoch, timeout_ns);
    // The list length is only known on the device, and a CTA without work still costs its launch.
    // A short list (the clones made private before the ray update, NVLink pulls) is bound by the dependent
    // round trips of its few items: more resident warps with fewer loads each (4 x 24 per SM) and one wave of
    // CTAs; the long list of eager copies prefers 8 x 12 (measured, profiles/r1_copy_tuning.md).
    if (short_list)
        k_copy_boxed<4, 24><<<num_sms * BOX_SHORT_CTAS, BOX_THREADS, 0, stream>>>(
            (const CopyJob*)jobs, leaders ? n_leaders : n_items, geom, counters);
    else
        k_copy_boxed<BOX_UNROLL, BOX_MINB><<<num_sms * BOX_CTAS_PER_SM, BOX_THREADS, 0, stream>>>(
            (const CopyJob*)jobs, leaders ? n_leaders : n_items, geom, counters);
}
size_t copy_job_bytes() { return sizeof(CopyJob); }

__global__ void k_commit_boxes(const CopyItem* __restrict__ items, const unsigned long long* __restrict__ n_items,
                               MapGeom geom, bool realign, StepCounters* counters, StepRecord* record,
                               StepCounters* host_mirror) {
    const unsigned long long n = *n_items;
    const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
    const unsigned long long tid = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    for (unsigned long long k = tid; k < n; k += stride) {
        *items[k].dst_meta = *items[k].src_meta;   // sources are never destinations of the same launch
    }
    if (!realign) {   // whole-grid copies moved the rows verbatim: the band tables go with them
        const uint32_t nb = bands_per_slot(geom);
        for (unsigned long long e = tid; e < n * nb; e += stride) {
            const unsigned long long k = e / nb;
            const uint32_t b = (uint32_t)(e - k * nb);
            items[k].dst_bands[b] = items[k].src_bands[b];
        }
    }
    if (record && blockIdx.x == 0 && threadIdx.x == 0) commit_step_record(counters, record);
    if (host_mirror != nullptr && blockIdx.x == 0) {
        __syncthreads();   // thread 0's est_box
        publish_mirror(counters, host_mirror);
    }
}
void launch_commit_boxes(cudaStream_t stream, const CopyItem* items, const unsigned long long* n_items, uint32_t max_items,
                         MapGeom geom, bool realign, StepCounters* counters, StepRecord* record, StepCounters* host_mirror) {
    const uint32_t blocks = realign ? (max_items + 255u) / 256u : 148u * 8u;
    k_commit_boxes<<<blocks ? blocks : 1, 256, 0, stream>>>(items, n_items, geom, realign, counters, record, host_mirror);
}

__global__ void k_account_full_copy(const unsigned long long* n_items, const unsigned long long* n_leaders,
                                    unsigned long long bytes_per_grid, StepCounters* counters) {
    counters->copy_bytes += bytes_per_grid * (*n_items + (n_leaders ? *n_leaders : *n_items));
}
void launch_account_full_copy(cudaStream_t stream, const unsigned long long* n_items, const unsigned long long* n_leaders,
                              size_t bytes_per_grid, StepCounters* counters) {
    k_account_full_copy<<<1, 1, 0, stream>>>(n_items, n_leaders, (unsigned long long)bytes_per_grid, counters);
}

}  // namespace slamrs
