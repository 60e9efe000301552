// The resampler up to the copy lists: k_weights (particle.rs:40-56, 59-65, 85-91), k_resample_indices
// (particle.rs:78-101) with the survivor list, k_mark_alive, k_plan (slot tables and copy items).
#include "kernels_common.cuh"

namespace slamrs {

// =============================================================================== k_weights

constexpr int W_CLUSTER = 8;   // largest (portable-size) thread-block cluster that shares the reduction

// ------------------------------------------------------------------------------- the exact left fold
// The reference adds weights strictly left to right (`iter().sum()`, particle.rs:50; `c += weight[i]`,
// particle.rs:91-93), and a resample threshold that lands within a few ulps of a prefix value selects a
// different particle if the sum is re-associated. The cluster reproduces the sequential fold bit for
// bit, in parallel (oracle/fold_model.py models the same steps on the CPU, tests/test_fold_model.py):
//
//  * While the running sum s stays inside one binade [2^e, 2^(e+1)], s = S * 2^(e-52) with S an integer
//    and fl(s + w) - s depends on s only through the parity of S (round-half-even ties). A chunk of
//    elements is therefore a two-state transducer: (d0, d1) = the total increment for an even / odd S at
//    entry, q = whether each flips the parity. Transducers compose associatively -> prefix scan.
//  * A chunk in which the sum changes binade is a "head": its output comes from a short sequential
//    chain over the heads (thread 0 of every CTA, operands prepared in shared memory by their owners).
//  * The binade of each chunk's incoming sum is GUESSED from an ordinary re-associated prefix sum. The
//    result is PROVED by induction: every thread folds its chunk from its incoming value with real
//    additions, and the outcome must equal, bit for bit, the incoming value its successor derived
//    independently through the scan. Everything in front of the first mismatch is proven; the
//    procedure restarts behind it from the now exact value (the "anchor"), which also settles on which
//    side of a binade edge a sum that creeps along the edge lies -- normalised weights end within a few
//    ulps of 1.0. After FOLD_MAX_ROUNDS rounds, or with more heads than the tables hold (NaN, inf,
//    adversarial inputs), thread 0 folds sequentially. Either way the result is the reference's.
//
// Shape (measured, profiles/r2_resample_exact.md): the kernel is bound by instruction issue -- every
// thread runs ~3,000 instructions of scans and bit tests whatever its chunk length -- so it uses few
// threads with long chunks: 512 threads x 16 elements per CTA, in registers, and as few CTAs as the
// population needs (one up to 8,192 particles: no cluster traffic at all).
constexpr uint32_t FOLD_HEADS_PER_CTA = 32;
constexpr uint32_t FOLD_HEADS_MAX = FOLD_HEADS_PER_CTA * W_CLUSTER;
constexpr uint32_t FOLD_STAGE = 2048;     // generic path: head operands staged in shared memory for the chain
constexpr int FOLD_MAX_ROUNDS = 4;
constexpr int FOLD_MARGIN_BITS = 40;      // "near a binade edge": within 2^-40 relative
constexpr int FOLD_LREG = 16;             // register path: elements per thread ...
constexpr int FOLD_THREADS = 512;         // ... and threads per CTA (up to 65,536 particles on 8 CTAs)
constexpr int FOLD_GENERIC_THREADS = 1024;
constexpr uint32_t FOLD_MAX_CHUNKS = FOLD_GENERIC_THREADS * W_CLUSTER;

struct FoldTd {       // transducer of a range of chunks; a range that contains a head forgets what precedes its last head
    double d0, d1;
    uint32_t qc;      // bits 0-1: parity flips for even / odd entry, bits 2..: heads in the range
};
template <int LREG>
struct FoldRec {      // one head, as the chain sees it
    double d0, d1;    // transducer of the regular chunks between the previous head of the same CTA (or the CTA's first chunk) and this one
    uint32_t q_prev;  // bits 0-1: q of that transducer, bit 2: an earlier head exists in the same CTA
    uint32_t chunk;
    double vals[LREG ? LREG : 1];   // the chunk's elements, zero-padded (register path)
};
template <int LREG>
struct FoldShared {
    double warp_f64[33];
    FoldTd warp_td[33];
    double cta_part[W_CLUSTER];                              // written by the peers (distributed shared memory)
    FoldTd cta_tot[W_CLUSTER];                               // "
    FoldRec<LREG> rec[W_CLUSTER][FOLD_HEADS_PER_CTA];        // "
    uint32_t cta_bad[W_CLUSTER];                             // "  first unproven chunk seen by each CTA
    uint32_t cta_overflow[W_CLUSTER];                        // "
    double total;                                            // "  the last chunk's outcome
    FoldTd cta_excl[W_CLUSTER + 1];                          // exclusive composition over the CTAs (local copy)
    double head_d0[FOLD_HEADS_MAX], head_d1[FOLD_HEADS_MAX]; // per head: the transducer in front of it, ready for the chain
    uint16_t head_rec[FOLD_HEADS_MAX];                       // per head: c * FOLD_HEADS_PER_CTA + k of its record
    double head_out[FOLD_HEADS_MAX];                         // the chain's results
    double vals[LREG ? 1 : FOLD_STAGE];                      // generic path: the heads' elements
    double warp_first[33];                                   // incoming value of each warp's first chunk
    uint32_t bad;                                            // this CTA's first unproven chunk
    uint32_t overflow;
};

__device__ __forceinline__ long long f64_bits(double x) { return __double_as_longlong(x); }
__device__ __forceinline__ int f64_exponent(double x) { return (int)((f64_bits(x) >> 52) & 0x7ff) - 1023; }
__device__ __forceinline__ double f64_pow2(int e) { return __longlong_as_double((long long)(e + 1023) << 52); }
__device__ __forceinline__ bool f64_finite(double x) { return ((f64_bits(x) >> 52) & 0x7ff) != 0x7ff; }

__device__ __forceinline__ FoldTd fold_compose(const FoldTd& a, const FoldTd& b) {
    FoldTd r;
    const uint32_t cnt = (a.qc >> 2) + (b.qc >> 2);
    if ((b.qc >> 2) != 0u) { r.d0 = b.d0; r.d1 = b.d1; r.qc = (b.qc & 3u) | (cnt << 2); return r; }
    const uint32_t p0 = a.qc & 1u;                    // parity after `a` for an even entry
    r.d0 = __dadd_rn(a.d0, p0 ? b.d1 : b.d0);
    const uint32_t q0 = p0 ^ ((b.qc >> p0) & 1u);
    const uint32_t a1 = (a.qc >> 1) & 1u;
    const uint32_t p1 = 1u ^ a1;                      // parity after `a` for an odd entry
    r.d1 = __dadd_rn(a.d1, p1 ? b.d1 : b.d0);
    const uint32_t q1 = a1 ^ ((b.qc >> p1) & 1u);
    r.qc = q0 | (q1 << 1) | (cnt << 2);
    return r;
}
__device__ __forceinline__ FoldTd fold_identity() { FoldTd t; t.d0 = 0.0; t.d1 = 0.0; t.qc = 0u; return t; }
__device__ __forceinline__ double fold_apply(const FoldTd& t, double s) {
    return __dadd_rn(s, (f64_bits(s) & 1ll) ? t.d1 : t.d0);
}
__device__ __forceinline__ FoldTd fold_shfl_up(const FoldTd& v, int o) {
    FoldTd r;
    r.d0 = __shfl_up_sync(0xffffffffu, v.d0, o);
    r.d1 = __shfl_up_sync(0xffffffffu, v.d1, o);
    r.qc = __shfl_up_sync(0xffffffffu, v.qc, o);
    return r;
}
// exclusive scan of one transducer per thread over the CTA (fold_compose is associative)
__device__ __forceinline__ FoldTd block_excl_scan_td(const FoldTd& v, FoldTd* warp_tot /*[33]*/, FoldTd* total) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    FoldTd inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const FoldTd t = fold_shfl_up(inc, o);
        if (lane >= o) inc = fold_compose(t, inc);
    }
    __syncthreads();
    if (lane == 31) warp_tot[wid] = inc;
    __syncthreads();
    if (wid == 0) {
        FoldTd winc = lane < nw ? warp_tot[lane] : fold_identity();
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const FoldTd t = fold_shfl_up(winc, o);
            if (lane >= o) winc = fold_compose(t, winc);
        }
        const FoldTd excl = fold_shfl_up(winc, 1);
        if (lane == 31) warp_tot[32] = winc;
        warp_tot[lane] = lane == 0 ? fold_identity() : excl;
    }
    __syncthreads();
    *total = warp_tot[32];
    const FoldTd within = fold_shfl_up(inc, 1);
    return lane == 0 ? warp_tot[wid] : fold_compose(warp_tot[wid], within);
}

// Binade the running sum is assumed to be in when the re-associated prefix says `a` (> 0, finite). Away
// from the binade edges: a's own. Within the margin of an edge 2^k (the top FOLD_MARGIN_BITS mantissa bits
// all 0 or all 1) the sum may be on either side: the side of the anchor (the last exactly known value) if
// the anchor lies in the same zone, else the lower one (a sum creeping up to an edge is below it until
// proven otherwise). *zone = near an edge.
__device__ __forceinline__ int fold_guess_binade(double a, double anchor, bool* zone) {
    const long long bits = f64_bits(a);
    const int e = (int)((bits >> 52) & 0x7ff) - 1023;
    const unsigned long long top = ((unsigned long long)bits & 0x000fffffffffffffull) >> (52 - FOLD_MARGIN_BITS);
    int k;
    if (top == 0ull) k = e;
    else if (top == (1ull << FOLD_MARGIN_BITS) - 1ull) k = e + 1;
    else { *zone = false; return e; }
    *zone = true;
    if (k < -960 || k > 1000) return k - 1;           // callers reject these exponents
    const double edge = f64_pow2(k);
    if (anchor > 0.0 && fabs(__dsub_rn(anchor, edge)) <= f64_pow2(k - FOLD_MARGIN_BITS)) return anchor >= edge ? k : k - 1;
    return k - 1;
}

struct FoldInfo { uint32_t rounds, heads, fallback; };
// SLAMRS_FOLD_TRACE: thread 0 of CTA 0 leaves clock64 stamps (tuning builds; SLAMRS_FOLD_TRACE_PRINT=1 prints them)
#ifdef SLAMRS_FOLD_TRACE
#define FOLD_STAMP(k) do { if (blockIdx.x == 0 && threadIdx.x == 0) reinterpret_cast<long long*>(g_fold_trace)[k] = clock64(); } while (0)
__device__ long long g_fold_trace[64];
#else
#define FOLD_STAMP(k) do { } while (0)
#endif

// barrier over the cluster; a single CTA needs no more than its own barrier
__device__ __forceinline__ void fold_sync(cg::cluster_group& cluster, uint32_t C) {
    if (C == 1u) __syncthreads(); else cluster.sync();
}

// One exact left fold over the cluster. The caller supplies this thread's chunk (L elements from index
// gt * L, `cnt` of them inside the population, through v[] (register path, zero-padded) or get_global(i))
// and a re-associated estimate (a_in0, a_out0) of the running sum in front of and behind the chunk. On
// return *s_in / *s_out hold the reference's running sum in front of / behind the chunk, put(j, s) has
// been called with the running sum after every element, *total is the grand total. Returns false if the
// fold could not be proven (too many heads, non-finite sums, rounds exhausted): the caller then folds
// sequentially. Cluster-uniform. scratch: 2 * FOLD_MAX_CHUNKS doubles.
template <int LREG, typename Put, typename GetGlobal>
__device__ bool exact_left_fold(cg::cluster_group& cluster, FoldShared<LREG>& sh, uint32_t n, uint32_t L, uint32_t cnt,
                                bool all_zero, double a_in0, double a_out0, const double (&v)[LREG ? LREG : 1], Put put,
                                GetGlobal get_global, bool first_is_assignment, double* __restrict__ scratch,
                                double* s_in_out, double* s_out_out, double* total, FoldInfo* info, int tb = 0) {
    (void)tb;
    const uint32_t crank = cluster.block_rank(), C = cluster.num_blocks();
    const uint32_t T = blockDim.x, tid = threadIdx.x, lane = tid & 31u, wid = tid >> 5;
    const uint32_t gt = crank * T + tid;
    const uint32_t lo = gt * L;
    const uint32_t last = (n - 1u) / L;               // last non-empty chunk (n >= 1)
    const bool assign_first = first_is_assignment && gt == 0u;
    double* __restrict__ sout = scratch;              // per chunk: the outcome of its fold (for the anchor)
    double* __restrict__ ain = scratch + FOLD_MAX_CHUNKS;   // per chunk: a_in0 (to re-base the estimate on the anchor)
    info->rounds = 0u; info->heads = 0u; info->fallback = 0u;
    ain[gt] = a_in0;

    uint32_t t0 = 0u;      // anchor: chunks < t0 are proven ...
    double s0 = 0.0;       // ... and s0 is the exact incoming value of chunk t0
    double a_base = 0.0;   // a_in0 of chunk t0
    for (int rnd = 0; rnd < FOLD_MAX_ROUNDS; ++rnd) {
        info->rounds = (uint32_t)rnd + 1u;
        if (tid == 0) { sh.bad = 0xffffffffu; sh.overflow = 0u; }
        const double a_in = rnd ? __dadd_rn(s0, __dsub_rn(a_in0, a_base)) : a_in0;
        const double a_out = rnd ? __dadd_rn(s0, __dsub_rn(a_out0, a_base)) : a_out0;
        // ---- 1. this chunk's transducer in the guessed binade
        FoldTd td = fold_identity();
        if (gt >= t0 && cnt != 0u && !all_zero) {        // (adding zeros changes nothing, whatever the binade)
            bool head = true;
            if (a_in > 0.0 && f64_finite(a_out)) {
                bool zone_in, zone_out;
                const int e = fold_guess_binade(a_in, s0, &zone_in);
                const int e_out = fold_guess_binade(a_out, s0, &zone_out);
                // regular: assumed to stay inside binade e. A chunk that enters an edge zone from outside is a head.
                if (e == e_out && (zone_in || !zone_out) && e >= -960 && e <= 1000) {
                    const double x0 = f64_pow2(e), x1 = __dadd_rn(x0, f64_pow2(e - 52));
                    double r0 = x0, r1 = x1;
                    if (LREG) {
#pragma unroll
                        for (int j = 0; j < (LREG ? LREG : 1); ++j) { r0 = __dadd_rn(r0, v[j]); r1 = __dadd_rn(r1, v[j]); }
                    } else {
                        for (uint32_t j = 0; j < cnt; ++j) { const double x = get_global(lo + j); r0 = __dadd_rn(r0, x); r1 = __dadd_rn(r1, x); }
                    }
                    if (r1 <= __dmul_rn(2.0, x0)) {
                        td.d0 = __dsub_rn(r0, x0); td.d1 = __dsub_rn(r1, x1);
                        td.qc = (uint32_t)(f64_bits(r0) & 1ll) | ((uint32_t)((f64_bits(r1) & 1ll) ^ 1ll) << 1);
                        head = false;
                    }
                }
            }
            if (head) td.qc = 1u << 2;
        }
        FOLD_STAMP(tb + 0);
        // ---- 2. scan; every head leaves a record in every CTA of the cluster
        FoldTd cta_total;
        const FoldTd excl = block_excl_scan_td(td, sh.warp_td, &cta_total);
        if ((td.qc >> 2) != 0u) {
            const uint32_t k = excl.qc >> 2;
            if (k >= FOLD_HEADS_PER_CTA) sh.overflow = 1u;
            else {
                for (uint32_t r = 0; r < C; ++r) {
                    FoldRec<LREG>* dst = C == 1u ? &sh.rec[0][k] : cluster.map_shared_rank(&sh.rec[0][0], r) + crank * FOLD_HEADS_PER_CTA + k;
                    dst->d0 = excl.d0; dst->d1 = excl.d1; dst->q_prev = (excl.qc & 3u) | (k ? 4u : 0u); dst->chunk = gt;
                    if (LREG) {
#pragma unroll
                        for (int j = 0; j < (LREG ? LREG : 1); ++j) dst->vals[j] = v[j];
                    }
                }
            }
        }
        FOLD_STAMP(tb + 1);
        __syncthreads();
        if (tid < C) {
            if (C == 1u) { sh.cta_tot[0] = cta_total; sh.cta_overflow[0] = sh.overflow; }
            else {
                cluster.map_shared_rank(&sh.cta_tot[0], tid)[crank] = cta_total;
                cluster.map_shared_rank(&sh.cta_overflow[0], tid)[crank] = sh.overflow;
            }
        }
        fold_sync(cluster, C);
        FOLD_STAMP(tb + 2);
        uint32_t overflow = 0u;
        for (uint32_t r = 0; r < C; ++r) overflow |= sh.cta_overflow[r];
        if (overflow) return false;                    // cluster-uniform
        // ---- 3. the chain over the heads (same computation in every CTA: no further exchange needed)
        if (tid == 0) {
            FoldTd run = fold_identity();
            for (uint32_t r = 0; r < C; ++r) { sh.cta_excl[r] = run; run = fold_compose(run, sh.cta_tot[r]); }
            sh.cta_excl[C] = run;
        }
        __syncthreads();
        const uint32_t H = sh.cta_excl[C].qc >> 2;
        for (uint32_t g = tid; g < H; g += T) {         // per head: where its record is and the transducer in front of it
            uint32_t c = 0u;
            while (c + 1u < C && (sh.cta_excl[c + 1u].qc >> 2) <= g) c++;
            const uint32_t k = g - (sh.cta_excl[c].qc >> 2);
            const FoldRec<LREG>& rec = sh.rec[c][k];
            FoldTd tail; tail.d0 = rec.d0; tail.d1 = rec.d1; tail.qc = rec.q_prev & 3u;
            if ((rec.q_prev & 4u) == 0u) tail = fold_compose(sh.cta_excl[c], tail);
            sh.head_d0[g] = tail.d0; sh.head_d1[g] = tail.d1;
            sh.head_rec[g] = (uint16_t)(c * FOLD_HEADS_PER_CTA + k);
        }
        bool staged = false;
        if (!LREG) {   // generic path: the heads' elements come from global memory, staged when they fit
            __syncthreads();
            staged = H * L <= FOLD_STAGE;
            if (staged)
                for (uint32_t j = tid; j < H * L; j += T) {
                    const uint32_t i = (&sh.rec[0][0])[sh.head_rec[j / L]].chunk * L + j % L;
                    sh.vals[j] = i < n ? get_global(i) : 0.0;
                }
        }
        __syncthreads();
        FOLD_STAMP(tb + 7);
        if (tid == 0) {
            double s = s0;
            for (uint32_t g = 0; g < H; ++g) {
                const FoldRec<LREG>& rec = (&sh.rec[0][0])[sh.head_rec[g]];
                s = __dadd_rn(s, (f64_bits(s) & 1ll) ? sh.head_d1[g] : sh.head_d0[g]);
                const bool assign = first_is_assignment && rec.chunk == 0u;
                if (LREG) {
                    s = assign ? rec.vals[0] : __dadd_rn(s, rec.vals[0]);
#pragma unroll
                    for (int j = 1; j < (LREG ? LREG : 1); ++j) s = __dadd_rn(s, rec.vals[j]);
                } else {
                    const uint32_t i0 = rec.chunk * L, m = min(n, i0 + L) - i0;
                    for (uint32_t j = 0; j < m; ++j) {
                        const double x = staged ? sh.vals[g * L + j] : get_global(i0 + j);
                        s = (assign && j == 0u) ? x : __dadd_rn(s, x);
                    }
                }
                sh.head_out[g] = s;
            }
            if (rnd == 0) info->heads = H;
        }
        FOLD_STAMP(tb + 3);
        __syncthreads();
        // ---- 4. every chunk: incoming value through the scan, real fold, comparison with the successor
        auto incoming = [&](const FoldTd& p) { return fold_apply(p, (p.qc >> 2) ? sh.head_out[(p.qc >> 2) - 1u] : s0); };
        const double s_in = incoming(fold_compose(sh.cta_excl[crank], excl));
        if (lane == 0) sh.warp_first[wid] = s_in;
        if (tid == 0) sh.warp_first[T >> 5] = incoming(sh.cta_excl[crank + 1u]);   // first chunk of the next CTA
        __syncthreads();
        FOLD_STAMP(tb + 4);
        double next_in = __shfl_down_sync(0xffffffffu, s_in, 1);
        if (lane == 31u) next_in = sh.warp_first[wid + 1u];
        if (gt >= t0 && gt <= last) {
            double s = s_in;
            if (LREG) {
                s = assign_first ? v[0] : __dadd_rn(s, v[0]);
                put(0, s);
#pragma unroll
                for (int j = 1; j < (LREG ? LREG : 1); ++j) { s = __dadd_rn(s, v[j]); if ((uint32_t)j < cnt) put(j, s); }
            } else {
                for (uint32_t j = 0; j < cnt; ++j) { const double x = get_global(lo + j); s = (assign_first && j == 0u) ? x : __dadd_rn(s, x); put(j, s); }
            }
            *s_in_out = s_in; *s_out_out = s;
            sout[gt] = s;
            if (gt < last && f64_bits(s) != f64_bits(next_in)) atomicMin(&sh.bad, gt + 1u);
            if (gt == last) {
                if (C == 1u) sh.total = s;
                else for (uint32_t r = 0; r < C; ++r) *cluster.map_shared_rank(&sh.total, r) = s;
            }
        }
        FOLD_STAMP(tb + 5);
        __syncthreads();
        if (tid < C) {
            if (C == 1u) sh.cta_bad[0] = sh.bad;
            else cluster.map_shared_rank(&sh.cta_bad[0], tid)[crank] = sh.bad;
        }
        fold_sync(cluster, C);    // (release / acquire at cluster scope: sout and ain of the other CTAs are visible)
        FOLD_STAMP(tb + 6);
        uint32_t bad = 0xffffffffu;
        for (uint32_t r = 0; r < C; ++r) bad = min(bad, sh.cta_bad[r]);
        if (bad == 0xffffffffu) { *total = sh.total; return true; }
        t0 = bad;
        s0 = __ldcg(&sout[bad - 1u]);                  // exact: every boundary in front of it matched
        a_base = __ldcg(&ain[bad]);
        if (!f64_finite(s0)) return false;             // NaN / inf: sequential
    }
    return false;
}

// normalize_weights (particle.rs:49-56), the argmax of particle.rs:40-46 and the running sum of
// particle.rs:85-91 over the WHOLE population, on one thread-block cluster of 1 to 8 CTAs; each thread
// owns a contiguous chunk of the population (in registers: LREG elements; LREG = 0: re-read from global
// memory, any length). Both sums are the reference's strict left folds (exact_left_fold); every GPU
// computes the same bits.
template <int LREG, int THREADS>
__global__ void __launch_bounds__(THREADS)
k_weights(const ParticleResult* __restrict__ results, uint32_t n, double* __restrict__ w_norm,
          double* __restrict__ cum, double* __restrict__ fold_scratch, double resample_tau, StepCounters* counters) {
    cg::cluster_group cluster = cg::this_cluster();
    const uint32_t crank = cluster.block_rank(), C = cluster.num_blocks();
    __shared__ FoldShared<LREG> sh;
    __shared__ double s_sq[W_CLUSTER];              // per-CTA sums of squared normalised weights (read by CTA 0)
    __shared__ long long s_key[32];
    __shared__ uint32_t s_arg[32];
    __shared__ long long s_ckey[W_CLUSTER];         // per-CTA argmax candidates (read by CTA 0)
    __shared__ uint32_t s_carg[W_CLUSTER];
    __shared__ double s_seq[2];
    pdl_launch_dependents();   // (k_resample_indices may become resident)
    pdl_wait();                // every weight of the step is in place (k_likelihood, or the barrier / all-gather behind it)
    FOLD_STAMP(0);
    const uint32_t gt = crank * THREADS + threadIdx.x;
    const uint32_t L = LREG ? (uint32_t)LREG : (n + C * THREADS - 1u) / (C * THREADS);
    const uint32_t lo = min(n, gt * L), hi = min(n, lo + L), cnt = hi - lo;

    // This thread's raw weights (zero-padded: adding +0.0 changes no non-negative sum). A thread owns LREG
    // consecutive elements, so direct accesses would touch 32 cache lines per warp instruction: loads and
    // stores go through a padded shared-memory tile instead, lanes striding over consecutive elements.
    extern __shared__ __align__(16) double s_tile[];   // register path: THREADS * (LREG + 1) doubles
    auto tile_of = [](uint32_t e) { return e + e / (uint32_t)(LREG ? LREG : 1); };
    const uint32_t warp_e0 = (threadIdx.x >> 5) * 32u * (uint32_t)(LREG ? LREG : 1);   // first element (within the CTA) of this warp
    const uint32_t cta_e0 = crank * THREADS * (uint32_t)(LREG ? LREG : 1);
    double v[LREG ? LREG : 1];
    double part = 0.0;
    bool all_zero = true;
    if (LREG) {
#pragma unroll
        for (int i = 0; i < (LREG ? LREG : 1); ++i) {
            const uint32_t e = warp_e0 + 32u * (uint32_t)i + (threadIdx.x & 31u);
            s_tile[tile_of(e)] = cta_e0 + e < n ? results[cta_e0 + e].weight : 0.0;
        }
        __syncwarp();
#pragma unroll
        for (int j = 0; j < (LREG ? LREG : 1); ++j) v[j] = s_tile[threadIdx.x * (LREG + 1) + j];
#pragma unroll
        for (int j = 0; j < (LREG ? LREG : 1); ++j) { part = __dadd_rn(part, v[j]); all_zero = all_zero && v[j] == 0.0; }
    } else {
        v[0] = 0.0;
        for (uint32_t j = 0; j < cnt; ++j) { const double x = results[lo + j].weight; part = __dadd_rn(part, x); all_zero = all_zero && x == 0.0; }
    }
    // the warp's LREG * 32 values of the tile -> dst, coalesced
    auto flush_tile = [&](double* __restrict__ dst) {
        __syncwarp();
#pragma unroll
        for (int i = 0; i < (LREG ? LREG : 1); ++i) {
            const uint32_t e = warp_e0 + 32u * (uint32_t)i + (threadIdx.x & 31u);
            if (cta_e0 + e < n) dst[cta_e0 + e] = s_tile[tile_of(e)];
        }
        __syncwarp();
    };
    if (gt == 0) {   // per-step counters start from zero
        counters->clamped = 0ull; counters->saturated = 0ull; counters->spilled = 0ull;
        counters->n_alive = 0ull; counters->copy_bytes = 0ull; counters->copy_max_rows = 0ull;
        counters->n_mat = 0ull; counters->n_mat_leaders = 0ull; counters->ray_cell_steps = 0ull; counters->ray_copy_bytes = 0ull;
        counters->ray_work_head = 0ull; counters->ray_items_front = 0ull; counters->ray_items_back = 0ull;
        counters->ray_items_front_local = 0ull; counters->ray_items_back_local = 0ull;
    }
    FOLD_STAMP(1);
    // re-associated prefix of the raw weights: the only ordinary scan of the kernel
    double cta_sum;
    const double offset = block_excl_scan_f64(part, sh.warp_f64, &cta_sum);
    double a_in = offset;
    if (C > 1u) {
        cluster.sync();   // every CTA of the cluster is running before its shared memory is written remotely
        if (threadIdx.x < C) cluster.map_shared_rank(&sh.cta_part[0], threadIdx.x)[crank] = cta_sum;
        cluster.sync();
        a_in = 0.0;
        for (uint32_t r = 0; r < crank; ++r) a_in = __dadd_rn(a_in, sh.cta_part[r]);
        a_in = __dadd_rn(a_in, offset);
    }
    const double a_out = __dadd_rn(a_in, part);
    FOLD_STAMP(2);

    // pass 1: sum of the raw weights, `self.weights.iter().sum()` (particle.rs:50)
    FoldInfo info_sum, info_cum;
    double r_in = 0.0, r_out = 0.0, sum = 0.0;
    bool ok = exact_left_fold<LREG>(cluster, sh, n, L, cnt, all_zero, a_in, a_out, v, [](uint32_t, double) {},
                                    [&](uint32_t i) { return results[i].weight; }, false, fold_scratch, &r_in, &r_out, &sum,
                                    &info_sum, 8);
    FOLD_STAMP(3);
    if (!ok) {   // the reference's loop as it stands, by one thread per CTA
        info_sum.fallback = 1u;
        if (threadIdx.x == 0) {
            double s = 0.0;
            for (uint32_t i = 0; i < n; ++i) s = __dadd_rn(s, results[i].weight);
            s_seq[0] = s;
        }
        __syncthreads();
        sum = s_seq[0];
    }

    // pass 2: normalise, argmax candidate, sum of squares
    double sqpart = 0.0;
    long long best_key = (long long)0x8000000000000000ull;
    uint32_t best_i = 0;
    bool have = false;
    all_zero = true;
    auto norm_one = [&](uint32_t j, double x) {
        const double w = __ddiv_rn(x, sum);
        if (LREG) s_tile[threadIdx.x * (LREG + 1) + j] = w; else w_norm[lo + j] = w;
        sqpart = __dadd_rn(sqpart, __dmul_rn(w, w));
        all_zero = all_zero && w == 0.0;
        const long long k = total_order_key(w);
        if (!have || k >= best_key) { best_key = k; best_i = lo + j; have = true; }  // last max wins
        return w;
    };
    if (LREG) {
#pragma unroll
        for (int j = 0; j < (LREG ? LREG : 1); ++j) v[j] = (uint32_t)j < cnt ? norm_one(j, v[j]) : 0.0;
        flush_tile(w_norm);
    } else {
        for (uint32_t j = 0; j < cnt; ++j) norm_one(j, results[lo + j].weight);
    }
    FOLD_STAMP(4);
    double cta_sq;
    const double sq_offset = block_excl_scan_f64(sqpart, sh.warp_f64, &cta_sq);

    // argmax by f64::total_cmp, ties -> highest index (Iterator::max_by returns the last maximum)
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    auto argmax_warp = [&]() {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const long long okey = __shfl_down_sync(0xffffffffu, best_key, o);
            const uint32_t oi = __shfl_down_sync(0xffffffffu, best_i, o);
            const bool ohave = __shfl_down_sync(0xffffffffu, (int)have, o) != 0;
            if (ohave && (!have || okey > best_key || (okey == best_key && oi > best_i))) { best_key = okey; best_i = oi; have = true; }
        }
    };
    argmax_warp();
    if (lane == 0) { s_key[wid] = best_key; s_arg[wid] = have ? best_i : 0xffffffffu; }
    __syncthreads();
    if (wid == 0) {
        have = lane < (THREADS >> 5) && s_arg[lane] != 0xffffffffu;
        best_key = have ? s_key[lane] : (long long)0x8000000000000000ull;
        best_i = have ? s_arg[lane] : 0u;
        argmax_warp();
        if (lane == 0) {
            if (C == 1u) { s_ckey[0] = best_key; s_carg[0] = have ? best_i : 0xffffffffu; s_sq[0] = cta_sq; }
            else {
                cluster.map_shared_rank(&s_ckey[0], 0)[crank] = best_key;
                cluster.map_shared_rank(&s_carg[0], 0)[crank] = have ? best_i : 0xffffffffu;
                cluster.map_shared_rank(&s_sq[0], 0)[crank] = cta_sq;
            }
        }
    }
    FOLD_STAMP(5);

    // pass 3: running sum of the normalised weights, `c = weights[0]; ... c += weights[i]` (particle.rs:85-93).
    // The exact raw prefixes of pass 1, divided by the sum, are the estimate that guesses the binades.
    if (ok) {
        double c_in, c_out, c_total;
        ok = exact_left_fold<LREG>(cluster, sh, n, L, cnt, all_zero, __ddiv_rn(r_in, sum), __ddiv_rn(r_out, sum), v,
                                   [&](uint32_t j, double s) { if (LREG) s_tile[threadIdx.x * (LREG + 1) + j] = s; else cum[lo + j] = s; },
                                   [&](uint32_t i) { return __ldcg(&w_norm[i]); }, true, fold_scratch, &c_in, &c_out, &c_total,
                                   &info_cum, 16);
        if (!ok) info_cum.fallback = 1u;
        else if (LREG) flush_tile(cum);
    } else {
        info_cum.rounds = 0u; info_cum.heads = 0u; info_cum.fallback = 1u;
    }
    FOLD_STAMP(6);
    if (!ok) {
        fold_sync(cluster, C);                          // every CTA's w_norm is written
        if (gt == 0) {
            double c = 0.0;
            for (uint32_t i = 0; i < n; ++i) { const double w = __ldcg(&w_norm[i]); c = i ? __dadd_rn(c, w) : w; cum[i] = c; }
        }
        fold_sync(cluster, C);
    }

    // pass 4, adaptive resampling only: the sum of squares of number_of_effective_particles (particle.rs:59-65),
    // `sum += w * w` left to right. N_eff < tau * N decides whether the filter resamples, and a re-associated sum
    // can land on the other side of tau * N than the reference's (equal weights at tau = 1: N_eff = N +- 1 ulp),
    // which changes the whole trajectory. The re-associated prefix of pass 2 is the estimate. With tau = 0 only
    // the reported N_eff depends on this sum, and the re-associated one is kept (no pass on the default path).
    FoldInfo info_sq = {0u, 0u, 0u};
    double sq_exact = 0.0;
    if (resample_tau > 0.0) {
        double q_in = sq_offset;
        if (C > 1u) {   // (every CTA has read sh.cta_part long before: pass 1 ended with cluster barriers)
            if (threadIdx.x < C) cluster.map_shared_rank(&sh.cta_part[0], threadIdx.x)[crank] = cta_sq;
            cluster.sync();
            q_in = 0.0;
            for (uint32_t r = 0; r < crank; ++r) q_in = __dadd_rn(q_in, sh.cta_part[r]);
            q_in = __dadd_rn(q_in, sq_offset);
        }
        if (LREG) {
#pragma unroll
            for (int j = 0; j < (LREG ? LREG : 1); ++j) v[j] = __dmul_rn(v[j], v[j]);   // (the padding stays +0.0)
        }
        double q_lo, q_hi;
        const bool sq_ok = exact_left_fold<LREG>(cluster, sh, n, L, cnt, all_zero, q_in, __dadd_rn(q_in, sqpart), v,
                                                 [](uint32_t, double) {},
                                                 [&](uint32_t i) { const double w = __ldcg(&w_norm[i]); return __dmul_rn(w, w); },
                                                 false, fold_scratch, &q_lo, &q_hi, &sq_exact, &info_sq, 24);
        if (!sq_ok) {   // the reference's loop as it stands (w_norm is complete: the fold passed cluster barriers)
            info_sq.fallback = 1u;
            if (gt == 0) {
                double s = 0.0;
                for (uint32_t i = 0; i < n; ++i) { const double w = __ldcg(&w_norm[i]); s = __dadd_rn(s, __dmul_rn(w, w)); }
                sq_exact = s;
            }
        }
    }
    // (a proven pass 3 ended with a cluster barrier: the peers' argmax candidates and sums of squares are in CTA 0)
    if (gt == 0) {
        long long bk = 0; uint32_t bi = 0; bool h = false;
        for (uint32_t r = 0; r < C; ++r) {
            if (s_carg[r] == 0xffffffffu) continue;
            if (!h || s_ckey[r] > bk || (s_ckey[r] == bk && s_carg[r] > bi)) { bk = s_ckey[r]; bi = s_carg[r]; h = true; }
        }
        counters->max_particle = bi;
        counters->sum = sum;
        // number_of_effective_particles (particle.rs:59-65) of the normalised weights, before resampling
        double sq = sq_exact;
        if (!(resample_tau > 0.0)) {
            sq = 0.0;
            for (uint32_t r = 0; r < C; ++r) sq = __dadd_rn(sq, s_sq[r]);
        }
        counters->n_eff = __ddiv_rn(1.0, sq);
        // adaptive resampling (not in the reference, which always resamples): only when N_eff < tau * N
        counters->do_resample = (resample_tau > 0.0 && !(__ddiv_rn(1.0, sq) < __dmul_rn(resample_tau, (double)n))) ? 0ull : 1ull;
        counters->fold_rounds = (unsigned long long)max(max(info_sum.rounds, info_cum.rounds), info_sq.rounds);
        counters->fold_heads = (unsigned long long)max(max(info_sum.heads, info_cum.heads), info_sq.heads);
        counters->fold_fallback = (unsigned long long)(info_sum.fallback | (info_cum.fallback << 1) | (info_sq.fallback << 2));
    }
    FOLD_STAMP(7);
}

static size_t weights_tile_bytes() { return sizeof(double) * FOLD_THREADS * (FOLD_LREG + 1); }
// cluster size by population: 512 threads x 16 elements per CTA, 1 / 2 / 4 / 8 CTAs up to 65,536 particles;
// beyond that the generic kernel (8 CTAs x 1024 threads, chunks of ceil(N / 8192) re-read from global memory)
WeightsShape weights_shape(uint32_t n_total) {
    uint32_t c = 1u;
    while (c < (uint32_t)W_CLUSTER && (uint64_t)c * FOLD_THREADS * FOLD_LREG < n_total) c <<= 1;
    WeightsShape s;
    s.cluster = c;
    s.regs = (uint64_t)c * FOLD_THREADS * FOLD_LREG >= n_total;
    s.threads = s.regs ? (uint32_t)FOLD_THREADS : (uint32_t)FOLD_GENERIC_THREADS;
    s.chunk = s.regs ? (uint32_t)FOLD_LREG : (uint32_t)(((uint64_t)n_total + c * s.threads - 1u) / (c * s.threads));
    return s;
}
void launch_weights(cudaStream_t stream, const ParticleResult* results, uint32_t n_total, double* w_norm,
                    double* cum, double* fold_scratch, double resample_tau, StepCounters* counters) {
    const WeightsShape shape = weights_shape(n_total);
    const uint32_t c = shape.cluster;
    const bool regs = shape.regs;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(c, 1, 1);
    cfg.blockDim = dim3(shape.threads, 1, 1);
    cfg.dynamicSmemBytes = regs ? weights_tile_bytes() : 0;
    cfg.stream = stream;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = c; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;   // (see launch_pdl)
    attr[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 2;
    if (regs) cudaLaunchKernelEx(&cfg, k_weights<FOLD_LREG, FOLD_THREADS>, results, n_total, w_norm, cum, fold_scratch, resample_tau, counters);
    else cudaLaunchKernelEx(&cfg, k_weights<0, FOLD_GENERIC_THREADS>, results, n_total, w_norm, cum, fold_scratch, resample_tau, counters);
}
size_t weights_scratch_doubles() { return 2u * FOLD_MAX_CHUNKS; }
int weights_trace(long long* out64) {
#ifdef SLAMRS_FOLD_TRACE
    return (int)cudaMemcpyFromSymbol(out64, g_fold_trace, sizeof(long long) * 64);
#else
    (void)out64;
    return -1;
#endif
}

// =============================================================================== k_resample_indices

// u_m of particle.rs:84, 89 for the zero-based new-particle index m0
__device__ __forceinline__ double resample_threshold(uint32_t n, double U, uint32_t m0) {
    const double num = (double)n;
    const double r = __ddiv_rn(__dmul_rn(U, 1.0), num);   // particle.rs:84: r = rand::random::<f64>() * 1.0 / N
    // particle.rs:89: u = r + (m as f64 - 1.0) * 1.0 / N with m = m0 + 1
    return __dadd_rn(r, __ddiv_rn(__dmul_rn(__dsub_rn((double)(m0 + 1u), 1.0), 1.0), num));
}
// first i in [lo, hi) with !(u > cum[i]), hi if none. particle.rs:91-94 advances i while u > c; c is
// non-decreasing (weights >= 0; NaN compares false from its first occurrence on), so the loop stops at
// the first i with !(u > cum[i]).
__device__ __forceinline__ uint32_t first_not_below(const double* __restrict__ cum, uint32_t lo, uint32_t hi, double u) {
    while (lo < hi) {
        const uint32_t mid = lo + ((hi - lo) >> 1);
        if (u > cum[mid]) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// Two-level search: a CTA first loads every RS_STRIDE-th running sum (the last of each block of RS_STRIDE
// weights, at most RS_COARSE of them) into shared memory in one round trip; a thread bisects there and
// finishes inside one block of the global array (one or two cache lines) instead of making log2(N)
// dependent trips to L2.
constexpr uint32_t RS_COARSE = 2048;

// Also builds the list of local particles that survive (some index selects them): a particle that
// no entry of the index vector selects is dropped by the resampler (particle.rs:88-104 builds the
// new generation only from old[i]); integrating the scan into its grid would be unobservable work,
// so the ray kernel runs on the survivors only. The thread of the FIRST new particle that selects a
// local source appends it (the index vector is non-decreasing, so "first" = differs from the
// predecessor's source, which comes from the neighbouring lane). With `ray` the survivors go straight
// into the fused ray update's work lists (kernels_ray.cu): a clone (grid still an alias of its source's
// slot) is listed in ray.clones, counts itself as a reader of its root and becomes private; a particle
// that owns its slot is listed in ray.owners.
__global__ void __launch_bounds__(256)
k_resample_indices(const ParticleResult* __restrict__ results, const double* __restrict__ cum, uint32_t n,
                   const double* __restrict__ u01_caller, uint64_t seed, uint64_t step, uint32_t* __restrict__ idx,
                   float* __restrict__ pose_next, uint32_t first_particle, uint32_t n_local, bool build_alive,
                   uint32_t* __restrict__ alive_list, RayLists ray, const double* __restrict__ w_norm,
                   double* __restrict__ carry, StepCounters* counters) {
    __shared__ double s_coarse[RS_COARSE];
    pdl_wait();                // k_weights has completed: normalised weights, running sum, counters
    const bool resample = counters->do_resample != 0ull;   // (adaptive resampling: 0 = every particle stays in place)
    const uint32_t stride = (n + RS_COARSE - 1u) / RS_COARSE;      // weights per block
    const uint32_t n_coarse = (n + stride - 1u) / stride;
    for (uint32_t j = threadIdx.x; j < n_coarse; j += blockDim.x) s_coarse[j] = cum[min(n, (j + 1u) * stride) - 1u];
    __syncthreads();
    const uint32_t m0 = blockIdx.x * blockDim.x + threadIdx.x;  // zero-based new-particle index
    const double U = u01_caller ? *u01_caller : slamrs_stream::resample_uniform(seed, step);
    const int lane = threadIdx.x & 31;
    auto source_of = [&](uint32_t m, bool* ran_off) {
        const double u = resample_threshold(n, U, m);
        const uint32_t blk = first_not_below(s_coarse, 0u, n_coarse, u);
        *ran_off = blk >= n_coarse;   // the reference would index out of bounds and panic; clamp and flag
        if (blk >= n_coarse) return n - 1u;
        return first_not_below(cum, blk * stride, min(n, (blk + 1u) * stride) - 1u, u);   // (the block's last element qualifies)
    };
    bool ran_off = false;
    uint32_t src_idx = 0xffffffffu;
    if (m0 < n) {
        if (resample) src_idx = source_of(m0, &ran_off); else src_idx = m0;
        if (carry != nullptr) carry[m0] = w_norm[m0];     // read by the next update only if this one did not resample
        if (m0 == 0u) counters->carry_active = resample ? 0ull : 1ull;
        if (ran_off) atomicAdd(&counters->clamped, 1ull);
        idx[m0] = src_idx;
        const ParticleResult src = results[src_idx];
        if (m0 >= first_particle && m0 < first_particle + n_local) {
            float* q = pose_next + 3 * (size_t)(m0 - first_particle);
            q[0] = src.x; q[1] = src.y; q[2] = src.theta;
        }
        // estimated_pose(), slam.rs:77-81: new generation indexed by the pre-resample argmax
        if ((unsigned long long)m0 == counters->max_particle) {
            counters->est_pose[0] = src.x; counters->est_pose[1] = src.y; counters->est_pose[2] = src.theta;
        }
    }
    if (!build_alive) return;   // uniform over the grid
    uint32_t prev = __shfl_up_sync(0xffffffffu, src_idx, 1);
    if (lane == 0 && m0 > 0 && m0 < n) {
        bool dummy;
        prev = resample ? source_of(m0 - 1u, &dummy) : m0 - 1u;
    }
    const bool alive = m0 < n && (m0 == 0 || prev != src_idx) && src_idx >= first_particle &&
                       src_idx < first_particle + n_local;
    // warp-aggregated appends (order is irrelevant: particles are independent)
    if (ray.clones == nullptr) {
        const unsigned mask = __ballot_sync(0xffffffffu, alive);
        if (mask) {
            const int leader = __ffs(mask) - 1;
            unsigned long long base = 0;
            if (lane == leader) base = atomicAdd(&counters->n_alive, (unsigned long long)__popc(mask));
            base = __shfl_sync(0xffffffffu, base, leader);
            if (alive) alive_list[base + __popc(mask & ((1u << lane) - 1u))] = src_idx - first_particle;
        }
        return;
    }
    RayItem it{0u, 0, 0, 0, 0, 0u};
    bool clone = false, remote = false;
    if (alive && ray.mark_remote != 0u) {
        // Does a new particle of another rank select this source (that rank pulls the grid in this step)? The index
        // vector is non-decreasing and this thread is the source's FIRST selector: either it belongs to another rank
        // itself, or the run of selectors reaches past the end of this rank's range.
        const uint32_t end = first_particle + n_local;
        remote = !(m0 >= first_particle && m0 < end);
        if (!remote && end < n) {
            bool dummy;
            remote = (resample ? source_of(end, &dummy) : end) == src_idx;
        }
    }
    if (alive) {
        it.pad = remote ? 1u : 0u;
        it.particle = src_idx - first_particle;
        it.slot = ray.slot_of[it.particle];
        it.root = ray.alias_of[it.slot];
        clone = it.root != it.slot;
        if (clone) {
            atomicAdd(&ray.readers[it.root], 2u);     // both halves of the clone read the root (k_ray_update_half)
            ray.alias_of[it.slot] = it.slot;
            // the slot takes its source's box now (the root's own update of it comes after its readers are done); what
            // the slot's previous tenant had informed still has to be cleared: the item remembers its rows
            const SlotMeta old = ray.meta[it.slot];
            if (old.x1 > old.x0 && old.y1 > old.y0) { it.old_y0 = old.y0; it.old_y1 = old.y1; }
            SlotMeta src = ray.meta[it.root];
            src.pad0 = 0;
            ray.meta[it.slot] = src;
        }
    }
    // four classes, in the order the ray update pops them: pulled clones, other clones, pulled owners, other owners
    // (a pulled grid is ready for its peer early; an owner still comes after every clone that reads its slot)
    const unsigned mcr = __ballot_sync(0xffffffffu, alive && clone && remote), mcl = __ballot_sync(0xffffffffu, alive && clone && !remote);
    const unsigned mor = __ballot_sync(0xffffffffu, alive && !clone && remote), mol = __ballot_sync(0xffffffffu, alive && !clone && !remote);
    unsigned long long bcr = 0, bcl = 0, bor = 0, bol = 0;
    if (lane == 0) {
        const unsigned mc = mcr | mcl, all = mc | mor | mol;
        if (all) atomicAdd(&counters->n_alive, (unsigned long long)__popc(all));
        if (mc) {
            atomicAdd(&counters->n_mat, (unsigned long long)__popc(mc));
            atomicAdd(&counters->n_mat_leaders, (unsigned long long)__popc(mc));   // every clone reads its source itself
        }
        if (mcr) bcr = atomicAdd(&counters->ray_items_front, (unsigned long long)__popc(mcr));
        if (mcl) bcl = atomicAdd(&counters->ray_items_front_local, (unsigned long long)__popc(mcl));
        if (mor) bor = atomicAdd(&counters->ray_items_back, (unsigned long long)__popc(mor));
        if (mol) bol = atomicAdd(&counters->ray_items_back_local, (unsigned long long)__popc(mol));
    }
    bcr = __shfl_sync(0xffffffffu, bcr, 0); bcl = __shfl_sync(0xffffffffu, bcl, 0);
    bor = __shfl_sync(0xffffffffu, bor, 0); bol = __shfl_sync(0xffffffffu, bol, 0);
    const unsigned below = (1u << lane) - 1u;
    if (alive && clone && remote) ray.clones[bcr + __popc(mcr & below)] = it;
    if (alive && clone && !remote) ray.clones[ray.n_local - 1u - (bcl + __popc(mcl & below))] = it;
    if (alive && !clone && remote) ray.owners[bor + __popc(mor & below)] = it;
    if (alive && !clone && !remote) ray.owners[ray.n_local - 1u - (bol + __popc(mol & below))] = it;
}

void launch_resample_indices(cudaStream_t stream, const ParticleResult* results, const double* cum,
                             uint32_t n_total, const double* u01_caller, uint64_t seed, uint64_t step,
                             uint32_t* idx, float* pose_next, uint32_t first_particle, uint32_t n_local,
                             bool build_alive, uint32_t* alive_list, RayLists ray, const double* w_norm, double* carry,
                             StepCounters* counters) {
    launch_pdl(k_resample_indices, dim3((n_total + 255) / 256), dim3(256), 0, stream, results, cum, n_total, u01_caller, seed, step, idx,
               pose_next, first_particle, n_local, build_alive, alive_list, ray, w_norm, carry, counters);
}

// =============================================================================== k_mark_alive
// The survivor list is normally built by k_resample_indices. This kernel builds it on its own:
// with all_particles the list is the identity (the reference's order of work: every particle's
// grid receives the scan).
__global__ void __launch_bounds__(256)
k_mark_alive(const uint32_t* __restrict__ idx, uint32_t n_total, uint32_t first_particle, uint32_t n_local,
             bool all_particles, uint32_t* __restrict__ alive_list, StepCounters* counters) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    bool alive = false;
    if (j < n_local) {
        if (all_particles) {
            alive = true;
        } else {
            const uint32_t v = first_particle + j;
            uint32_t lo = 0, hi = n_total;
            while (lo < hi) {
                const uint32_t mid = lo + ((hi - lo) >> 1);
                if (idx[mid] < v) lo = mid + 1; else hi = mid;
            }
            alive = lo < n_total && idx[lo] == v;
        }
    }
    // warp-aggregated append (order is irrelevant: particles are independent)
    const unsigned m = __ballot_sync(0xffffffffu, alive);
    if (m) {
        const int lane = threadIdx.x & 31, leader = __ffs(m) - 1;
        unsigned long long base = 0;
        if (lane == leader) base = atomicAdd(&counters->n_alive, (unsigned long long)__popc(m));
        base = __shfl_sync(0xffffffffu, base, leader);
        if (alive) alive_list[base + __popc(m & ((1u << lane) - 1u))] = j;
    }
}

void launch_mark_alive(cudaStream_t stream, const uint32_t* idx, uint32_t n_total, uint32_t first_particle,
                       uint32_t n_local, bool all_particles, uint32_t* alive_list, StepCounters* counters) {
    k_mark_alive<<<(n_local + 255) / 256, 256, 0, stream>>>(idx, n_total, first_particle, n_local, all_particles,
                                                           alive_list, counters);
}

// =============================================================================== k_plan
// Turns the (non-decreasing) index vector into work for this rank's output range [lo, lo+S):
//   0  source is local and this is its first use here   -> the grid stays where it is
//   1  source is local, further use                     -> copy from the kept grid into a free slot
//   2  source lives on another GPU, first use here      -> copy over NVLink into a free slot
//   3  source lives on another GPU, further use         -> likewise (every 16th use re-reads the source)
// All copies form ONE list in output order; copies of one source are adjacent, and every
// COPY_FAN-th of them is a "leader": the copy kernel reads the source once per leader and stores it
// to the whole sub-run. Free slots = slots of local particles nobody here keeps + the persistent
// spare slots. A dropped slot whose grid another GPU copies from in this step ("unsafe") is not
// handed out now -- it joins the spare list of the next step -- so no rank ever writes a grid
// that a peer may still be reading, and one cross-GPU barrier per resampling is enough. That needs
// n_unsafe <= n_spare; otherwise the step reports SLAMRS_E_STAGING (raise spare_slots).

__device__ __forceinline__ uint32_t lower_bound_u32(const uint32_t* a, uint32_t lo, uint32_t hi, uint32_t v) {
    while (lo < hi) {
        const uint32_t mid = lo + ((hi - lo) >> 1);
        if (a[mid] < v) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// With n_local <= PLAN_STAGED_MAX_S the index range, the slot tables, the class bytes and the free
// list live in shared memory (22 bytes per particle): the planner is a chain of short sequential
// passes whose cost is load latency, and shared memory cuts that by an order of magnitude.
constexpr uint32_t PLAN_STAGED_MAX_S = 8192;
__host__ __device__ inline size_t plan_staged_bytes(uint32_t S) { return (size_t)S * 22u + 64u; }

__global__ void __launch_bounds__(1024) k_plan(PlanArgs a) {
    extern __shared__ __align__(16) unsigned char s_dyn[];
    __shared__ uint32_t s_warp[33];
    const uint32_t S = a.n_local, lo = a.rank * a.n_local, hi = lo + S;
    const uint32_t T = blockDim.x, t = threadIdx.x;
    const uint32_t chunk = (S + T - 1) / T;
    const uint32_t c0 = min(S, t * chunk), c1 = min(S, c0 + chunk);
    const uint32_t E = (uint32_t)a.counters->n_spare;

    // working arrays: shared memory when staged, the global scratch otherwise
    uint32_t* idx_l;       // idx[lo .. hi)
    int32_t* slot_old;     // read-only copy
    int32_t* slot_new;
    int32_t* free_list;    // [safe | spare | unsafe]
    uint8_t* keep;
    uint8_t* need;
    if (a.staged) {
        idx_l = reinterpret_cast<uint32_t*>(s_dyn);
        slot_old = reinterpret_cast<int32_t*>(idx_l + S);
        slot_new = slot_old + S;
        free_list = slot_new + S;          // 2 S + 1 entries (E <= S when staged)
        keep = reinterpret_cast<uint8_t*>(free_list + 2 * (size_t)S + 4);
        need = keep + S;
        for (uint32_t j = t; j < S; j += T) { idx_l[j] = a.idx[lo + j]; slot_old[j] = a.slot_old[j]; keep[j] = 0; }
    } else {
        idx_l = const_cast<uint32_t*>(a.idx) + lo;
        slot_old = const_cast<int32_t*>(a.slot_old);
        slot_new = a.slot_new;
        free_list = a.free_list;
        keep = reinterpret_cast<uint8_t*>(a.keep);
        need = reinterpret_cast<uint8_t*>(a.need);
        for (uint32_t j = t; j < S; j += T) keep[j] = 0;
    }
    __syncthreads();

    // ---- classify new particles
    uint32_t nA = 0, nR = 0;
    for (uint32_t m = t; m < S; m += T) {
        const uint32_t src = idx_l[m];
        const bool first = (m == 0) || (idx_l[m - 1] != src);
        const bool local = (src >= lo && src < hi);
        int cls;
        if (local && first) {
            cls = 0;
            keep[src - lo] = 1;
            slot_new[m] = slot_old[src - lo];
        } else if (local) cls = 1;
        else if (first) cls = 2;
        else cls = 3;
        need[m] = (uint8_t)cls;
        nA += (first ? 1u : 0u);
        nR += (cls == 2 ? 1u : 0u);
    }
    __syncthreads();

    // ---- classify old slots: 0 = kept, 1 = free & safe, 2 = free but read by another GPU this step.
    // A slot that is not kept has no local consumer; idx is non-decreasing, so its consumers (if
    // any) are all before this rank's range (v < idx[lo]) or all after it (v > idx[hi-1]).
    const uint32_t idx_first = idx_l[0], idx_last = idx_l[S - 1];
    for (uint32_t j = t; j < S; j += T) {
        int f = 0;
        if (!keep[j]) {
            f = 1;
            if (a.world > 1) {
                const uint32_t v = lo + j;
                if (v < idx_first && lo > 0) {
                    const uint32_t p = lower_bound_u32(a.idx, 0, lo, v);
                    if (p < lo && a.idx[p] == v) f = 2;
                } else if (v > idx_last && hi < a.n_total) {
                    const uint32_t p = lower_bound_u32(a.idx, hi, a.n_total, v);
                    if (p < a.n_total && a.idx[p] == v) f = 2;
                }
            }
        }
        keep[j] = (uint8_t)f;
    }
    __syncthreads();

    // ---- ordered compaction of the free slots: [safe | spare | unsafe]
    uint32_t n_safe_c = 0, n_unsafe_c = 0;
    for (uint32_t j = c0; j < c1; ++j) { n_safe_c += (keep[j] == 1); n_unsafe_c += (keep[j] == 2); }
    uint32_t n_safe, n_unsafe;
    uint32_t ps = block_excl_scan_u32(n_safe_c, s_warp, &n_safe);
    uint32_t pu = block_excl_scan_u32(n_unsafe_c, s_warp, &n_unsafe);
    for (uint32_t j = c0; j < c1; ++j) {
        if (keep[j] == 1) free_list[ps++] = slot_old[j];
        else if (keep[j] == 2) free_list[n_safe + E + pu++] = slot_old[j];
    }
    for (uint32_t e = t; e < E; e += T) free_list[n_safe + e] = a.spare_list[e];
    const uint32_t usable = n_safe + E;   // slots that may be written in this step

    // ---- ordered ranks of the consumers (every new particle that does not keep a grid in place)
    // Every consumer takes a free slot. Eager: every consumer is also a copy. Deferred: only the first
    // local use of a remote source is copied (over NVLink, after the barrier); every other consumer
    // becomes an alias of its source's slot (PlanArgs::alias_of) and moves no bytes now.
    uint32_t n_cons_c = 0, n_item_c = 0;
    for (uint32_t m = c0; m < c1; ++m) { n_cons_c += (need[m] != 0); n_item_c += (need[m] == 2); }
    uint32_t n_cons, n_items = 0;
    uint32_t pos = block_excl_scan_u32(n_cons_c, s_warp, &n_cons);
    uint32_t ipos = a.defer ? block_excl_scan_u32(n_item_c, s_warp, &n_items) : pos;   // position in copies[]
    __syncthreads();  // free_list complete

    // ---- the copy list. run_first = first position of the current source's run in this range.
    const uint32_t ipos_start = ipos;
    uint32_t n_lead_c = 0;
    const unsigned long long est_m = a.counters->max_particle - lo;   // >= S when another rank owns the estimate
    if (t == 0 && est_m >= S) a.counters->est_meta_ptr = 0ull;
    uint32_t run_first = c0 < c1 ? lower_bound_u32(idx_l, 0, S, idx_l[c0]) : 0u;
    for (uint32_t m = c0; m < c1; ++m) {
        const int cls = need[m];
        const uint32_t src = idx_l[m];
        if (m > c0 && idx_l[m - 1] != src) run_first = m;
        if (cls == 0) {
            // the published map (slam.rs:83-88) is this particle's grid: it stays in place
            if (m == est_m) a.counters->est_meta_ptr = (unsigned long long)(uintptr_t)(a.meta + slot_new[m]);
            continue;
        }
        if (pos < usable && a.defer && cls != 2) {
            slot_new[m] = free_list[pos];
            need[m] = (uint8_t)(cls == 1 ? 11 : 12);   // alias of a local source / of this rank's copy of a remote one
            if (m == est_m && cls == 1) a.counters->est_meta_ptr = (unsigned long long)(uintptr_t)(a.meta + slot_old[src - lo]);
        } else if (pos < usable) {
            const int32_t dslot = free_list[pos];
            slot_new[m] = dslot;
            CopyItem it;
            if (cls == 1) {
                const int32_t sslot = slot_old[src - lo];
                it.src = a.cells + (size_t)sslot * a.cells_per_grid;
                it.src_meta = a.meta + sslot;
                it.src_bands = a.bands + (size_t)sslot * a.n_bands;
            } else {
                const uint32_t owner = src / S;
                const int32_t sslot = a.results[src].slot;
                it.src = a.peer_cells[owner] + (size_t)sslot * a.cells_per_grid;
                it.src_meta = a.peer_meta[owner] + sslot;
                it.src_bands = a.peer_bands[owner] + (size_t)sslot * a.n_bands;
            }
            it.dst = a.cells + (size_t)dslot * a.cells_per_grid;
            it.dst_meta = a.meta + dslot;
            it.dst_bands = a.bands + (size_t)dslot * a.n_bands;
            a.copies[ipos] = it;
            if (m == est_m) a.counters->est_meta_ptr = (unsigned long long)(uintptr_t)it.src_meta;   // extent it will have
            // a local run keeps its first use in place, so its copies start one position later
            const uint32_t k = (cls == 1) ? (m - run_first - 1u) : (m - run_first);
            const bool lead = a.defer || (k % COPY_FAN) == 0u;
            need[m] = (uint8_t)(lead ? 9 : 8);
            n_lead_c += lead;
            if (a.defer) ipos++;
        } else {
            // no writable slot left (SLAMRS_E_STAGING): nothing is copied, the filter state is invalid
            slot_new[m] = (cls == 1) ? slot_old[src - lo] : slot_old[0];
            need[m] = 10;
        }
        pos++;
        if (!a.defer) ipos = pos;
    }
    // ordered list of leader positions within copies[]
    uint32_t n_lead;
    uint32_t pl = block_excl_scan_u32(n_lead_c, s_warp, &n_lead);
    ipos = ipos_start;
    for (uint32_t m = c0; m < c1; ++m) {
        const int cls = need[m];
        if (cls == 9) a.leaders[pl++] = ipos;
        if (cls == 8 || cls == 9 || (!a.defer && cls == 10)) ipos++;
    }
    __syncthreads();   // slot_new complete
    // ---- deferred copies: the new particle's slot stands for its source's slot until it is written
    long long est_root = -1ll;
    if (a.defer) {
        for (uint32_t m = c0; m < c1; ++m) {
            const int cls = need[m];
            int32_t root = slot_new[m];
            if (cls == 11) root = slot_old[idx_l[m] - lo];
            else if (cls == 12) root = slot_new[lower_bound_u32(idx_l, 0, S, idx_l[m])];   // this rank's first use: the copy
            if (cls == 8 || cls == 9 || cls == 11 || cls == 12) a.alias_of[slot_new[m]] = root;
            if (m == est_m) {
                est_root = root;
                if (cls == 12) a.counters->est_meta_ptr = (unsigned long long)(uintptr_t)(a.meta + root);
            }
        }
        if (est_root >= 0) a.counters->est_slot = est_root;   // the published map is read from the cells it shares
    }
    __syncthreads();
    // ---- next step's spare list: the usable slots nobody took, then this step's unsafe slots
    const uint32_t used = min(n_cons, usable);
    for (uint32_t e = t; e < E; e += T) {
        const uint32_t left = usable - used;   // = E - n_unsafe when nothing is short
        a.spare_list[e] = e < left ? free_list[used + e] : free_list[usable + (e - left)];
    }
    if (a.staged)
        for (uint32_t m = t; m < S; m += T) a.slot_new[m] = slot_new[m];

    uint32_t distinct, n_remote;
    block_excl_scan_u32(nA, s_warp, &distinct);
    block_excl_scan_u32(nR, s_warp, &n_remote);
    if (t == 0) {
        // staging short: positions in copies[] have holes (consumers without a slot), so the list is not
        // handed to the copy kernels at all -- the step fails with SLAMRS_E_STAGING and copies nothing
        const bool short_of_slots = n_cons > usable;
        const uint32_t n_copied = a.defer ? n_items : used;
        a.counters->n_copies = short_of_slots ? 0u : n_copied;
        a.counters->n_leaders = short_of_slots ? 0u : n_lead;
        a.counters->n_pulls = n_remote;
        a.counters->distinct = distinct;
        a.counters->staging_short = (n_cons > usable) ? (unsigned long long)(n_cons - usable) : 0ull;
        const unsigned long long mp = a.counters->max_particle;
        a.counters->est_owner = mp / S;
        if (!a.defer || !(mp >= lo && mp < hi))   // deferred: set above by the thread that owns the estimate
            a.counters->est_slot = (mp >= lo && mp < hi) ? (long long)slot_new[mp - lo] : -1ll;
        if (a.history) {
            StepRecord r;
            r.step = a.step; r.n_copies = n_copied; r.n_pulls = n_remote; r.distinct = distinct; r.n_leaders = n_lead;
            r.n_alive = 0; r.copy_bytes = 0; r.ray_cell_steps = 0; r.ray_copy_bytes = 0;   // filled in by the step's last kernel (k_commit_boxes)
            a.history[a.step % STEP_HISTORY] = r;
        }
    }
}

// =============================================================================== k_materialize_list
// exclusive running maximum of one uint32 per thread over a 1024-thread CTA (0 = nothing before)
__device__ __forceinline__ uint32_t block_excl_scan_max_u32(uint32_t v, uint32_t* warp_tot /*[33]*/) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    uint32_t inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc = max(inc, t);
    }
    __syncthreads();  // protect warp_tot reuse across calls
    if (lane == 31) warp_tot[wid] = inc;
    __syncthreads();
    if (wid == 0) {
        const uint32_t w = lane < nw ? warp_tot[lane] : 0u;
        uint32_t winc = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, winc, o);
            if (lane >= o) winc = max(winc, t);
        }
        const uint32_t excl = __shfl_up_sync(0xffffffffu, winc, 1);
        warp_tot[lane] = lane == 0 ? 0u : excl;   // maximum over the earlier warps
    }
    __syncthreads();
    const uint32_t within = __shfl_up_sync(0xffffffffu, inc, 1);
    return max(warp_tot[wid], lane == 0 ? 0u : within);
}

// A clone that resampling created is an alias of its source's slot until somebody writes it
// (PlanArgs::alias_of). The particles whose grids this step writes -- the local particles the index
// vector selects, or all of them -- get their own cells first: one CopyItem (root slot -> own slot)
// per shared grid, in particle order. Clones of one source are neighbours in that order, so the
// fan-out leaders are found as in k_plan: the head of each run of equal roots and every COPY_FAN-th
// item after it. One CTA: the work is three short ordered passes over n_local entries.
__global__ void __launch_bounds__(1024)
k_materialize_list(const uint32_t* __restrict__ idx, uint32_t n_total, uint32_t first_particle, uint32_t S,
                   const int32_t* __restrict__ slot_of, int32_t* alias_of, uint32_t* cells, size_t cells_per_grid,
                   SlotMeta* meta, uint32_t* bands, uint32_t n_bands, CopyItem* __restrict__ items,
                   uint32_t* __restrict__ leaders, uint32_t* roots, StepCounters* counters) {
    __shared__ uint32_t s_warp[33];
    const uint32_t T = blockDim.x, t = threadIdx.x;
    const uint32_t chunk = (S + T - 1) / T;
    const uint32_t c0 = min(S, t * chunk), c1 = min(S, c0 + chunk);
    auto shared_and_written = [&](uint32_t j, int32_t* slot, int32_t* root) {
        if (idx != nullptr) {   // is local particle j selected by the index vector?
            const uint32_t v = first_particle + j;
            const uint32_t q = lower_bound_u32(idx, 0, n_total, v);
            if (q >= n_total || idx[q] != v) return false;
        }
        *slot = slot_of[j];
        *root = alias_of[*slot];
        return *root != *slot;
    };
    uint32_t cnt = 0;
    int32_t slot, root;
    for (uint32_t j = c0; j < c1; ++j) cnt += shared_and_written(j, &slot, &root) ? 1u : 0u;
    uint32_t total;
    uint32_t pos = block_excl_scan_u32(cnt, s_warp, &total);
    for (uint32_t j = c0; j < c1; ++j) {
        if (!shared_and_written(j, &slot, &root)) continue;
        CopyItem it;
        it.src = cells + (size_t)root * cells_per_grid;
        it.src_meta = meta + root;
        it.src_bands = bands + (size_t)root * n_bands;
        it.dst = cells + (size_t)slot * cells_per_grid;
        it.dst_meta = meta + slot;
        it.dst_bands = bands + (size_t)slot * n_bands;
        items[pos] = it;
        roots[pos] = (uint32_t)root;
        alias_of[slot] = slot;   // private from here on (the copy is issued right after this kernel)
        pos++;
    }
    __syncthreads();
    // leaders: run heads and every COPY_FAN-th item of a run
    const uint32_t ichunk = (total + T - 1) / T;
    const uint32_t i0 = min(total, t * ichunk), i1 = min(total, i0 + ichunk);
    uint32_t last_head = 0u;   // position + 1 of the last run head in this thread's items
    for (uint32_t i = i0; i < i1; ++i)
        if (i == 0u || roots[i] != roots[i - 1u]) last_head = i + 1u;
    const uint32_t before = block_excl_scan_max_u32(last_head, s_warp);
    uint32_t run_start = before ? before - 1u : 0u, n_lead_c = 0u;
    for (uint32_t i = i0; i < i1; ++i) {
        if (i == 0u || roots[i] != roots[i - 1u]) run_start = i;
        n_lead_c += ((i - run_start) % COPY_FAN) == 0u;
    }
    uint32_t n_lead;
    uint32_t pl = block_excl_scan_u32(n_lead_c, s_warp, &n_lead);
    run_start = before ? before - 1u : 0u;
    for (uint32_t i = i0; i < i1; ++i) {
        if (i == 0u || roots[i] != roots[i - 1u]) run_start = i;
        if (((i - run_start) % COPY_FAN) == 0u) leaders[pl++] = i;
    }
    if (t == 0) { counters->n_mat = total; counters->n_mat_leaders = n_lead; }
}

// The common case (survivors only): the survivor list is a few hundred entries long and already on the
// device, so the shared grids among them are listed by one thread per survivor, in no particular order
// and without fan-out grouping (every item reads its own source; the list is short).
__global__ void __launch_bounds__(256)
k_materialize_alive(const uint32_t* __restrict__ alive_list, const int32_t* __restrict__ slot_of, int32_t* alias_of,
                    uint32_t* cells, size_t cells_per_grid, SlotMeta* meta, uint32_t* bands, uint32_t n_bands,
                    CopyItem* __restrict__ items, StepCounters* counters) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    bool take = false;
    int32_t slot = 0, root = 0;
    if ((unsigned long long)i < counters->n_alive) {
        slot = slot_of[alive_list[i]];
        root = alias_of[slot];
        take = root != slot;
    }
    const unsigned mask = __ballot_sync(0xffffffffu, take);
    if (mask == 0u) return;
    const int lane = threadIdx.x & 31, leader = __ffs(mask) - 1;
    unsigned long long base = 0;
    if (lane == leader) {
        base = atomicAdd(&counters->n_mat, (unsigned long long)__popc(mask));
        atomicAdd(&counters->n_mat_leaders, (unsigned long long)__popc(mask));   // every item reads its source itself
    }
    base = __shfl_sync(0xffffffffu, base, leader);
    if (!take) return;
    CopyItem it;
    it.src = cells + (size_t)root * cells_per_grid;
    it.src_meta = meta + root;
    it.src_bands = bands + (size_t)root * n_bands;
    it.dst = cells + (size_t)slot * cells_per_grid;
    it.dst_meta = meta + slot;
    it.dst_bands = bands + (size_t)slot * n_bands;
    items[base + __popc(mask & ((1u << lane) - 1u))] = it;
    alias_of[slot] = slot;
}
void launch_materialize_alive(cudaStream_t stream, const uint32_t* alive_list, uint32_t n_local, const int32_t* slot_of,
                              int32_t* alias_of, uint32_t* cells, size_t cells_per_grid, SlotMeta* meta, uint32_t* bands,
                              uint32_t n_bands, CopyItem* items, StepCounters* counters) {
    k_materialize_alive<<<(n_local + 255) / 256, 256, 0, stream>>>(alive_list, slot_of, alias_of, cells, cells_per_grid, meta,
                                                                   bands, n_bands, items, counters);
}

void launch_materialize_list(cudaStream_t stream, const uint32_t* idx, uint32_t n_total, uint32_t first_particle,
                             uint32_t n_local, const int32_t* slot_of, int32_t* alias_of, uint32_t* cells,
                             size_t cells_per_grid, SlotMeta* meta, uint32_t* bands, uint32_t n_bands, CopyItem* items,
                             uint32_t* leaders, uint32_t* roots_scratch, StepCounters* counters) {
    k_materialize_list<<<1, 1024, 0, stream>>>(idx, n_total, first_particle, n_local, slot_of, alias_of, cells, cells_per_grid,
                                               meta, bands, n_bands, items, leaders, roots_scratch, counters);
}

bool plan_can_stage(uint32_t n_local, uint32_t n_spare_cap) {
    return n_local <= PLAN_STAGED_MAX_S && n_spare_cap <= n_local;
}

void launch_plan(cudaStream_t stream, const PlanArgs& a) {
    k_plan<<<1, 1024, a.staged ? plan_staged_bytes(a.n_local) : 0, stream>>>(a);
}

cudaError_t configure_resample_kernels() {
    cudaError_t e = cudaFuncSetAttribute(k_weights<FOLD_LREG, FOLD_THREADS>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)weights_tile_bytes());
    if (e != cudaSuccess) return e;
    return cudaFuncSetAttribute(k_plan, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)plan_staged_bytes(PLAN_STAGED_MAX_S));
}

}  // namespace slamrs
