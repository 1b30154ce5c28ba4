// bdg_join.cuh -- edge construction at t = 2 and t = 3 by sort-merge joins on multi-block seeds (bdg_seed.cuh, bdg_seed3.cuh); sm_100a.
// Reference semantics: index.py:77-93 (candidate filter S >= T) + barcode_graph.py:233-249 (3-way edit-distance verify, emit).
//
// Per condition c of the seed scheme the N barcodes are bucketed by the condition's join key (the kernels read a key off a
// barcode in a few shifts and masks, so only the barcodes are stored), once as rows
// (fields of x) and - for the conditions with a shifted diagonal - once as columns (the matching fields of y).  Equal keys
// are then adjacent on both sides: row i pairs with the column run colstart[key(i)] .. colstart[key(i) + 1].
//   join_hist_rank_kernel / join_scatter_rank_kernel  counting sort by the join key (one digit; cub's scan turns the bucket
//                          sizes into colstart, the first column of every key value) with one atomic per barcode: the counting
//                          pass keeps the place its atomic returned.
//   join_band_kernel<T>    per slab of 32 consecutive rows: number of work units (runs of <= JUNIT columns) it needs
//   (cub::DeviceScan::ExclusiveSum: unit index -> slab)
//   join_kernel<T, RS, SHF> one persistent launch per condition: warps pull batches of units from an atomic cursor, stage the
//                          unit's columns in their own slice of shared memory (y, y >> 2, y << 2, key) and test
//                          (row, column) pairs: quick test of bdg_core.cuh + key equality, one hit bit per pair; hits go
//                          through the warp's queue to the exact stage on full warps, edges are appended with one atomic per warp.
// A unit's 32 rows are worked through as 32/RS sub-slabs of RS rows x 32/RS column phases, each against its own column run:
// RS = 32 when the key buckets are long, RS = 8 when they are short (fewer rows span fewer foreign buckets).
// What differs between the thresholds T is the per-pair stage:
//   T = 2  quick test on ONE diagonal side (join2_quick, bdg_seed.cuh), two marks dropped: a shifted condition (SHF) tests the
//          row's side {0, +1} and stages no y << 2, a symmetric one passes a pair on {0, +1} or on {0, -1}; exact stage
//          join_process: dist_small, the hand-over table over seed_flags and the two side bits (seed_side_bits) on full batches
//          of close pairs, then the 6-mer score in two queues (the middle diagonals, then the other eighteen).
//   T = 3  quick test on the diagonals -2..2 (quick3_marks; the +-2 words are derived from the staged +-1 ones), three marks
//          dropped; exact stage join3_process: dist3_min (Myers' bit-vector pass; D <= 3 has no case analysis), the hand-over
//          walk seed3_first, then the 6-mer score through one queue.  The t = 3 scheme is too large for constant memory next to
//          the t = 2 one: the kernels read the condition's two keys from their arguments and the hand-over tables from a device
//          copy of the Seed3Scheme.
// The conditions are dealt to the parts (GPUs / ranks) by estimated work (join_weigh_*, join3_weigh_*), a condition on a part
// boundary is split by row range at a bucket boundary (join_cut), so a part sorts only the conditions it works on.  No
// block-level barrier anywhere.
#pragma once
#include <type_traits>
#include "bdg_edges.cuh"
#include "bdg_seed.cuh"
#include "bdg_seed3.cuh"

namespace bdg {

constexpr int JCH = 128;           // columns staged at a time
constexpr int JPAD = 32;           // slack behind the staged columns (steps may start up to one step early)
constexpr int JUNIT = 2048;        // columns per work unit
constexpr int JBATCH = 4;          // units per cursor fetch
constexpr int JQCAP = 120;         // candidate queue entries per warp (with the other arrays: 5 CTAs of 8 warps per SM at t = 2)
constexpr int JQ2CAP = 64;         // entries of each exact-stage queue (t = 2: close pairs and two scoring queues; t = 3: one scoring queue)
constexpr int JROWS = 32;          // rows per slab
// edge-count snapshots of the streaming form: one after every condition at t = 2, one after every block set at t = 3
constexpr int JOIN_MAX_SNAPS = SEED_MAX_CONDS > SEED3_MAX_SETS ? SEED_MAX_CONDS : SEED3_MAX_SETS;

__constant__ SeedScheme c_scheme;

#ifdef BDG_JOIN_LANE_STATS
// Development build (make EXTRA=-DBDG_JOIN_LANE_STATS; read with bdg_join_lane_stats): how full the warps of the candidate push and
// of the exact stages run.  [0] push rounds, [1] hits pushed, [2] candidate batches through dist_small, [3] their candidates,
// [4] of those batches, the ones with a pair at D <= 2, [5] batches through the hand-over check, [6] their pairs.
__device__ unsigned long long g_join_lane[8];
#define BDG_LANE_ADD(k, v)                                                                                           \
    do {                                                                                                             \
        const unsigned long long v_ = (unsigned long long)(v);                                                      \
        if ((threadIdx.x & 31) == 0) atomicAdd(&g_join_lane[k], v_);                                                 \
    } while (0)
#else
#define BDG_LANE_ADD(k, v) do { } while (0)
#endif

struct JoinArgs {
    const uint32_t* rows;          // barcodes in the order of the row-side key of the condition
    const uint32_t* cols;          // ... of the column-side key (== rows for a symmetric condition)
    const uint32_t* colstart;      // (1 << key_bits) + 1 lower bounds into cols
    const uint32_t* offs;          // exclusive prefix sums of the units per slab: n_slabs + 1 entries
    const uint8_t* lut;            // t = 2: hand-over table over seed_flags
    unsigned long long* cursor;    // batches handed out by this launch
    unsigned long long* stats;     // [0] units, [2] pairs tested, [3] candidates, [6] pairs with D <= t, [7] of those owned and scored, [4]/[5] warp times
    uint32_t N, n_slabs;
    int cond, self;
    const uint32_t* rowstart;      // (1 << key_bits) + 1 lower bounds into rows (== colstart for a symmetric condition)
    uint32_t nkeys;
    uint32_t f0, f1, fden;         // this part works on the rows [cut(f0), cut(f1)) of the condition: cuts at bucket boundaries near N * f / fden
    int T;
    uint32_t one, mone;            // runtime 1 / -1: u * one + mone is u - 1 on the FMA pipe
};

// t = 3: the keys and the hand-over tables travel with the launch (the t = 2 ones sit in c_scheme)
struct Join3Args : JoinArgs {
    SeedKey ka, kb;                // the condition's row-side / column-side key
    const Seed3Scheme* scheme;     // device copy: hand-over tables
};

template <int T>
using JoinArgsT = std::conditional_t<T == 2, JoinArgs, Join3Args>;

template <int T>
__device__ __forceinline__ const SeedKey& join_ka(const JoinArgsT<T>& A)
{
    if constexpr (T == 2) return c_scheme.ka[A.cond]; else return A.ka;
}

template <int T>
__device__ __forceinline__ const SeedKey& join_kb(const JoinArgsT<T>& A)
{
    if constexpr (T == 2) return c_scheme.kb[A.cond]; else return A.kb;
}

// ---- bucketing by join key: a counting sort in three launches (the key has <= 20 bits, so ONE digit: no radix passes) ----
//   join_hist_rank_kernel     bucket sizes (one global atomic per barcode; the 2^key_bits counters stay in L2); each barcode
//                             keeps what its atomic returned, its place inside its bucket
//   (cub::DeviceScan::ExclusiveSum over the counters: colstart, the first position of every key value)
//   join_scatter_rank_kernel  every barcode to start[key] + place
// The order inside a bucket is whatever the atomics give: the join pairs whole buckets, so it does not matter.
__global__ void join_hist_rank_kernel(const uint32_t* __restrict__ in, uint32_t n, SeedKey k, uint32_t* __restrict__ hist, uint32_t* __restrict__ rank)
{
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) rank[i] = atomicAdd(&hist[seed_key(__ldg(&in[i]), k)], 1u);
}

__global__ void join_scatter_rank_kernel(const uint32_t* __restrict__ in, uint32_t n, SeedKey k, const uint32_t* __restrict__ start,
                                         const uint32_t* __restrict__ rank, uint32_t* __restrict__ out)
{
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const uint32_t v = __ldg(&in[i]);
        out[__ldg(&start[seed_key(v, k)]) + __ldg(&rank[i])] = v;
    }
}

// Where a part's share of a condition starts / ends: the first row of the first bucket that begins at or behind N * f / fden.
// Bucket boundaries depend on the bucket SIZES only, so every part finds the same cut whatever order its own counting sort
// left inside the buckets, and a bucket is never split between parts.
__device__ __forceinline__ uint32_t join_cut(const uint32_t* __restrict__ rowstart, uint32_t nkeys, uint32_t N, uint32_t f, uint32_t fden)
{
    if (f == 0) return 0u;
    if (f >= fden) return N;
    const uint32_t target = (uint32_t)((uint64_t)N * f / fden);
    uint32_t lo = 0, hi = nkeys;                          // smallest key whose bucket starts at or behind the target (rowstart[nkeys] = N)
    while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        if (__ldg(&rowstart[mid]) < target) lo = mid + 1; else hi = mid;
    }
    return __ldg(&rowstart[lo]);
}

// ---- how much work is a condition?  (the deal of the conditions to several parts) -------------------------------------
// Bucket sizes of every condition over a SAMPLE of the barcodes (every stride-th one): the number of (row, column) pairs a
// condition has to test is sum_k rows_k * cols_k (a symmetric one: sum_k n_k (n_k - 1) / 2), and the sample's sum times
// stride^2 estimates it.  Integer counts over the same sample on every part, so every part computes the same deal.
// t = 2 samples all its tables in one pass; t = 3 goes block set by block set, because its 475 tables do not fit at once.
struct WeighSlots { uint8_t row[SEED_MAX_CONDS], col[SEED_MAX_CONDS]; int n; };   // table of a condition's row / column key (a block set shares its row table)

__global__ void join_weigh_hist_kernel(const uint32_t* __restrict__ in, uint32_t n, uint32_t stride, int nconds, uint32_t tab, const WeighSlots ws,
                                       uint32_t* __restrict__ hist)
{
    const uint32_t m = (n + stride - 1) / stride;
    for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; j < m; j += gridDim.x * blockDim.x) {
        const uint32_t x = __ldg(&in[(uint64_t)j * stride]);
        for (int c = 0; c < nconds; c++) {
            if (c_scheme.cond[c].row_sort == c) atomicAdd(&hist[(size_t)ws.row[c] * tab + seed_key(x, c_scheme.ka[c])], 1u);
            if (!c_scheme.cond[c].self) atomicAdd(&hist[(size_t)ws.col[c] * tab + seed_key(x, c_scheme.kb[c])], 1u);
        }
    }
}

// grid (x, nconds): condition blockIdx.y, four counters per thread and step
__global__ void join_weigh_sum_kernel(const uint32_t* __restrict__ hist, uint32_t tab, const WeighSlots ws, unsigned long long* __restrict__ out)
{
    const int c = blockIdx.y;
    const bool self = c_scheme.cond[c].self != 0;
    const uint4* __restrict__ hr = reinterpret_cast<const uint4*>(hist + (size_t)ws.row[c] * tab);
    const uint4* __restrict__ hc = reinterpret_cast<const uint4*>(hist + (size_t)ws.col[c] * tab);
    unsigned long long mine = 0;
    for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < tab / 4; k += gridDim.x * blockDim.x) {
        const uint4 r = __ldg(&hr[k]);
        if (self) {
            mine += (unsigned long long)r.x * (r.x - (r.x ? 1 : 0)) / 2 + (unsigned long long)r.y * (r.y - (r.y ? 1 : 0)) / 2 +
                    (unsigned long long)r.z * (r.z - (r.z ? 1 : 0)) / 2 + (unsigned long long)r.w * (r.w - (r.w ? 1 : 0)) / 2;
        } else if (r.x | r.y | r.z | r.w) {
            const uint4 q = __ldg(&hc[k]);
            mine += (unsigned long long)r.x * q.x + (unsigned long long)r.y * q.y + (unsigned long long)r.z * q.z + (unsigned long long)r.w * q.w;
        }
    }
    for (int o = 16; o; o >>= 1) mine += __shfl_down_sync(FULL, mine, o);
    if ((threadIdx.x & 31) == 0 && mine) atomicAdd(&out[c], mine);
}

// Work estimate of the t = 3 conditions c0 .. c1 - 1 of one block set: table 0 holds the row key of the set (its first,
// symmetric, condition), table c - c0 the column key of condition c.
__global__ void join3_weigh_hist_kernel(const uint32_t* __restrict__ in, uint32_t n, uint32_t stride, const Seed3Scheme* __restrict__ S, int c0, int c1,
                                        uint32_t tab, uint32_t* __restrict__ hist)
{
    const uint32_t m = (n + stride - 1) / stride;
    for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; j < m; j += gridDim.x * blockDim.x) {
        const uint32_t x = __ldg(&in[(uint64_t)j * stride]);
        atomicAdd(&hist[seed_key(x, S->ka[c0])], 1u);
        for (int c = c0 + 1; c < c1; c++) atomicAdd(&hist[(size_t)(c - c0) * tab + seed_key(x, S->kb[c])], 1u);
    }
}

// grid (x, c1 - c0): pairs of condition c0 + blockIdx.y over the sample
__global__ void join3_weigh_sum_kernel(const uint32_t* __restrict__ hist, uint32_t tab, int c0, unsigned long long* __restrict__ out)
{
    const int q = blockIdx.y;
    const uint32_t* __restrict__ hr = hist;
    const uint32_t* __restrict__ hc = hist + (size_t)q * tab;
    unsigned long long mine = 0;
    for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < tab; k += gridDim.x * blockDim.x) {
        const unsigned long long r = __ldg(&hr[k]);
        if (q == 0) mine += r * (r - (r ? 1 : 0)) / 2;
        else if (r) mine += r * __ldg(&hc[k]);
    }
    for (int o = 16; o; o >>= 1) mine += __shfl_down_sync(FULL, mine, o);
    if ((threadIdx.x & 31) == 0 && mine) atomicAdd(&out[c0 + q], mine);
}

// the edge count as it stands when the stream reaches this point (bdg_edges_build_into copies the finished edges out meanwhile)
__global__ void join_snapshot_kernel(const unsigned long long* __restrict__ count, volatile unsigned long long* __restrict__ snap)
{
    *snap = *count;
}

// units of every slab of 32 rows: its column run (first key's bucket .. last key's bucket; a symmetric condition pairs
// each couple once - column index > row index - so its run starts behind the slab's first row) in pieces of JUNIT columns
template <int T>
__global__ void join_band_kernel(const JoinArgsT<T> A, uint32_t* __restrict__ counts)
{
    const SeedKey& ka = join_ka<T>(A);
    const uint32_t r0 = join_cut(A.rowstart, A.nkeys, A.N, A.f0, A.fden), r1 = join_cut(A.rowstart, A.nkeys, A.N, A.f1, A.fden);
    for (uint32_t s = blockIdx.x * blockDim.x + threadIdx.x; s <= A.n_slabs; s += gridDim.x * blockDim.x) {
        uint32_t cnt = 0;
        if (s < A.n_slabs) {
            const uint32_t i0 = max(s * JROWS, r0), i1 = min(min(A.N, s * JROWS + JROWS), r1);      // the slab's rows of this part: [i0, i1)
            if (i0 < i1) {
                uint32_t lo = __ldg(&A.colstart[seed_key(__ldg(&A.rows[i0]), ka)]);
                const uint32_t hi = __ldg(&A.colstart[seed_key(__ldg(&A.rows[i1 - 1u]), ka) + 1u]);
                if (A.self) lo = max(lo, i0 + 1u);
                cnt = hi > lo ? (hi - lo + JUNIT - 1) / JUNIT : 0u;
            }
        }
        counts[s] = cnt;
    }
}

struct JoinCtx {
    uint2* q;                      // candidates (x, y): row value, column value
    uint2* q2;                     // (a, b) with D <= t owned by this pass that still need the 6-mer score
    uint8_t* q2d;
    const uint8_t* lut;            // t = 2: hand-over table
    int lane, T, cond, shifted;    // shifted: 1 for a condition with a shifted diagonal (its two value orders are two hand-over indices)
    unsigned long long n_near, n_owned;   // pairs with D <= t; of those, owned by this pass and handed to the score
    const Seed3Scheme* scheme;     // t = 3: hand-over tables
};

// t = 2 exact stage: three stages chained by per-warp queues in q2 / q2d, each run on full batches of 32 only (except the flush):
//   candidates (one per lane) -> dist_small -> pairs with D <= 2 into the close-pair queue;
//   32 close pairs -> seed_flags + hand-over table -> pairs this pass owns into the scoring queue;
//   32 owned pairs -> 6-mer score of the middle diagonals; the undecided wait for the other eighteen in a second scoring queue.
// Only about a quarter of the candidates are close: behind its own queue the hand-over check runs on full warps instead of on
// every candidate batch that holds one close pair (nearly all of them).
// Every queue holds fewer than 32 entries when a stage starts and a stage adds at most 32, so JQ2CAP = 64 entries never overflow.
// A real call, not inlined: one copy of the exact distance and of the score loop keeps the kernel's hot code inside the instruction
// cache (ncu: the fully inlined form spent most of its issue slots waiting for instructions).  Everything travels in registers:
// q2n packs the three fills (JFILL_BITS each, see below); returns the new fills | pairs with D <= 2 << 16 | pairs handed to the
// score << 24.
// want0 / want1: the hand-over index this pass owns for a candidate with row value < / > column value (the same for a symmetric
// condition, whose buckets are in no particular order).  flush: run the hand-over check on a partial batch of close pairs (the end
// of a launch; no candidates then).
constexpr int JFILL_BITS = 5;      // a queue fill between calls is < 32
constexpr int JQ_NEAR = 0, JQ_FAR = JQ2CAP, JQ_CLOSE = 2 * JQ2CAP;   // t = 2: the three queues of q2 / q2d

__device__ __forceinline__ int jfill(int q2n, int k) { return (q2n >> (k * JFILL_BITS)) & ((1 << JFILL_BITS) - 1); }

__device__ __noinline__ uint32_t join_process(uint2* q2, uint8_t* q2d, const uint8_t* lut, int want0, int want1, int T, const EdgeOut out, uint2 e, bool active,
                                              int q2n, bool flush)
{
    // q2 holds three queues: entries [JQ_NEAR, +64) owned pairs that still need their score, [JQ_FAR, +64) pairs whose three middle
    // diagonals did not reach the threshold and need the other eighteen, [JQ_CLOSE, +64) pairs with D <= 2 before the hand-over check
    const int lane = threadIdx.x & 31;
    const unsigned lt = (1u << lane) - 1u;
    int n1 = jfill(q2n, 0), n2 = jfill(q2n, 1), nc = jfill(q2n, 2);
    const uint32_t a = min(e.x, e.y), b = max(e.x, e.y);
    bool ok = active && a != b;
    int d = 3;
    if (ok) { d = dist_small(a, b, false, true); ok = d <= 2; }
    const unsigned mc = __ballot_sync(FULL, ok);
    if (ok) {                                            // D (1 or 2) and the orientation: want0 / want1 depend on the original order
        const int slot = JQ_CLOSE + nc + __popc(mc & lt);
        q2[slot] = make_uint2(a, b);
        q2d[slot] = (uint8_t)(d | (e.x > e.y ? 4 : 0));
    }
    nc += __popc(mc);
    if (!flush) { BDG_LANE_ADD(2, 1); BDG_LANE_ADD(3, __popc(__ballot_sync(FULL, active))); BDG_LANE_ADD(4, mc != 0); }
    uint32_t n_own = 0;
    if (nc >= 32 || (flush && nc > 0)) {                 // hand-over check on a full batch of close pairs
        __syncwarp();
        const int take = min(nc, 32);
        nc -= take;
        bool own = false;
        uint2 v = make_uint2(0u, 0u);
        uint8_t vd = 0;
        if (lane < take) {
            v = q2[JQ_CLOSE + nc + lane];
            vd = q2d[JQ_CLOSE + nc + lane];
            const uint32_t idx = seed_flags(c_scheme, v.x, v.y) | seed_side_bits(v.x, v.y) << c_scheme.nflags;
            own = __ldg(&lut[idx]) == (uint8_t)((vd & 4) ? want1 : want0);   // emitted by the first (condition, orientation) that meets and passes the pair
        }
        const unsigned m = __ballot_sync(FULL, own);
        n_own = (uint32_t)__popc(m);
        BDG_LANE_ADD(5, 1); BDG_LANE_ADD(6, take);
        if (own) {
            const int slot = JQ_NEAR + n1 + __popc(m & lt);
            q2[slot] = v;
            q2d[slot] = (uint8_t)(vd & 3);
        }
        n1 += __popc(m);
        __syncwarp();
        if (n1 >= 32) {                                  // full batch: score of the middle diagonals; what they decide is emitted
            n1 -= 32;
            const uint2 mv = q2[JQ_NEAR + n1 + lane];
            const uint8_t md = q2d[JQ_NEAR + n1 + lane];
            const int near = qgram_score_near(mv.x, mv.y);
            emit_warp(near >= T, mv.x, mv.y, md, out);
            const unsigned rest = __ballot_sync(FULL, near < T);
            if (near < T) {
                const int slot = JQ_FAR + n2 + __popc(rest & lt);
                q2[slot] = mv;
                q2d[slot] = (uint8_t)(md | (near << 2));     // distance (1 or 2) and the part of the score that is known
            }
            n2 += __popc(rest);
            __syncwarp();
            if (n2 >= 32) {                              // a full batch of the undecided: the other eighteen diagonals
                n2 -= 32;
                const uint2 fv = q2[JQ_FAR + n2 + lane];
                const uint8_t fd = q2d[JQ_FAR + n2 + lane];
                emit_warp((int)(fd >> 2) + qgram_score_far(fv.x, fv.y) >= T, fv.x, fv.y, fd & 3, out);
                __syncwarp();
            }
        }
    }
    return (uint32_t)(n1 | (n2 << JFILL_BITS) | (nc << (2 * JFILL_BITS))) | ((uint32_t)__popc(mc) << 16) | (n_own << 24);
}

// t = 3 exact stage on a batch of candidates (one per lane): D, hand-over walk, survivors into the scoring queue, full batches of
// that queue through the 6-mer score.  Not inlined, as at t = 2: one copy of the bit-vector pass, the walk and the score loop.
// The walk runs after the distance, on the candidates within D <= 3 only (DESIGN.md 3.8).
// Returns the queue fill | pairs with D <= 3 << 16 | pairs owned by this pass << 24, the packing of join_process.
__device__ __noinline__ uint32_t join3_process(uint2* q2, uint8_t* q2d, const Seed3Scheme* S, int want0, int want1, int T, const EdgeOut out,
                                               uint2 e, bool active, int n1)
{
    const int lane = threadIdx.x & 31;
    const uint32_t a = min(e.x, e.y), b = max(e.x, e.y);
    const int want = e.x > e.y ? want1 : want0;
    bool ok = active && a != b;
    int d = 4;
    if (ok) { d = dist3_min(a, b); ok = d <= 3; }
    const uint32_t n_d3 = (uint32_t)__popc(__ballot_sync(FULL, ok));
    if (ok) ok = seed3_first(*S, a, b) == want;          // emitted by the first (condition, orientation) the pair meets
    const uint32_t n_own = (uint32_t)__popc(__ballot_sync(FULL, ok));
    const unsigned m = __ballot_sync(FULL, ok);
    if (m) {
        if (ok) {                                        // fewer than 32 entries wait on entry, so 32 more always fit
            const int slot = n1 + __popc(m & ((1u << lane) - 1u));
            q2[slot] = make_uint2(a, b);
            q2d[slot] = (uint8_t)d;
        }
        n1 += __popc(m);
        __syncwarp();
        if (n1 >= 32) {
            n1 -= 32;
            const uint2 v = q2[n1 + lane];
            const uint8_t vd = q2d[n1 + lane];
            emit_warp(qgram_score_compact(v.x, v.y) >= T, v.x, v.y, vd, out);
            __syncwarp();
        }
    }
    return (uint32_t)n1 | (n_d3 << 16) | (n_own << 24);
}

template <int T>
__device__ __forceinline__ void join_drain(JoinCtx& c, const EdgeOut& out, int& qn, int& q2n, bool all)
{
    __syncwarp();
    while (qn >= 32 || (all && qn > 0)) {
        const int take = min(qn, 32);
        qn -= take;
        const uint2 e = c.lane < take ? c.q[qn + c.lane] : make_uint2(0u, 0u);
        uint32_t r;
        if constexpr (T == 2) r = join_process(c.q2, c.q2d, c.lut, 2 * c.cond, 2 * c.cond + c.shifted, c.T, out, e, c.lane < take, q2n, false);
        else r = join3_process(c.q2, c.q2d, c.scheme, 2 * c.cond, 2 * c.cond + c.shifted, c.T, out, e, c.lane < take, q2n);
        q2n = (int)(r & 0xFFFFu);
        c.n_near += (r >> 16) & 255u;
        c.n_owned += r >> 24;
        __syncwarp();
    }
    if constexpr (T == 2) {
        if (all) {                                       // the close pairs still waiting: a partial batch through the hand-over check
            const uint32_t r = join_process(c.q2, c.q2d, c.lut, 2 * c.cond, 2 * c.cond + c.shifted, c.T, out, make_uint2(0u, 0u), false, q2n, true);
            q2n = (int)(r & 0xFFFFu);
            c.n_owned += r >> 24;
            __syncwarp();
        }
    }
}

// append the hits of a group of 8 steps: bit 4 * st + kk of h = column colbase + st * STEP + kk of the staged sub-tile
template <int T, int STEP>
__device__ __forceinline__ void join_push(uint32_t h, uint32_t x, const uint32_t* sb0, int colbase, int& qn, int& q2n, JoinCtx& c, const EdgeOut& out)
{
    const int cnt = __popc(h);
    int incl = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(FULL, incl, o);
        if (c.lane >= o) incl += v;
    }
    const int total = __shfl_sync(FULL, incl, 31);
    if (qn + total <= JQCAP) {
        BDG_LANE_ADD(0, __reduce_max_sync(FULL, (unsigned)cnt)); BDG_LANE_ADD(1, total);
        int slot = qn + incl - cnt;
        while (h) {
            const int j = __ffs(h) - 1;
            h &= h - 1;
            c.q[slot++] = make_uint2(x, sb0[colbase + (j >> 2) * STEP + (j & 3)]);
        }
        qn += total;
        join_drain<T>(c, out, qn, q2n, false);
        return;
    }
    for (;;) {                                           // burst larger than the queue: one hit per lane and round
        const bool has = h != 0;
        const unsigned m = __ballot_sync(FULL, has);
        if (m == 0) break;
        BDG_LANE_ADD(0, 1); BDG_LANE_ADD(1, __popc(m));
        if (has) {
            const int j = __ffs(h) - 1;
            h &= h - 1;
            c.q[qn + __popc(m & ((1u << c.lane) - 1u))] = make_uint2(x, sb0[colbase + (j >> 2) * STEP + (j & 3)]);
        }
        qn += __popc(m);                                 // qn < 32 before every round, so the round's <= 32 entries fit
        join_drain<T>(c, out, qn, q2n, false);
    }
}

// T = 2 is compiled for 5 resident CTAs per SM (48 registers; its three exact-stage queues take 41 KB of shared memory per CTA),
// T = 3 for 4: its exact stage needs the registers.
// SHF (T = 2 only): a launch of a shifted condition, whose pairs are tested on the one diagonal side {0, +1} of the row
// (join2_quick<true>; the y << 2 words are neither staged nor read); the symmetric conditions test either side.  T = 3 keeps
// the test on -2..2 and the symmetric / shifted split at run time.
template <int T, int RS, bool SHF = false>
__global__ void __launch_bounds__(ENT, T == 2 ? 5 : 4) join_kernel(const JoinArgsT<T> A, const EdgeOut out)
{
    static_assert(T == 2 || !SHF, "the one-sided test is the t = 2 one");
    constexpr int PH = 32 / RS;                          // column phases of a warp
    constexpr int STEP = 4 * PH;                         // columns per inner step
    __shared__ __align__(16) uint32_t s_b[EW][4][JCH + JPAD];   // y, y >> 2, y << 2 (not for SHF), key of the staged columns
    __shared__ uint2 s_q[EW][JQCAP];
    __shared__ uint2 s_q2[EW][T == 2 ? 3 * JQ2CAP : JQ2CAP];   // pairs that need their score | (t = 2) pairs that need the far diagonals | close pairs
    __shared__ uint8_t s_q2d[EW][T == 2 ? 3 * JQ2CAP : JQ2CAP];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int r = lane & (RS - 1), ph = lane / RS;
    uint32_t* const sb0 = s_b[wid][0];
    uint32_t* const sbP = s_b[wid][1];
    uint32_t* const sbM = s_b[wid][2];
    uint32_t* const sbK = s_b[wid][3];
    JoinCtx c;
    c.q = s_q[wid]; c.q2 = s_q2[wid]; c.q2d = s_q2d[wid];
    if constexpr (T == 2) c.lut = A.lut; else c.scheme = A.scheme;
    c.lane = lane; c.T = A.T; c.cond = A.cond; c.shifted = A.self ? 0 : 1; c.n_near = 0; c.n_owned = 0;
    int qn = 0, q2n = 0;
    const uint32_t mone = A.mone;
    const unsigned long long t_start = global_ns();
    unsigned long long n_units = 0, n_pairs = 0, n_cand = 0;
    const SeedKey& ka = join_ka<T>(A);
    const SeedKey& kb = join_kb<T>(A);
    const bool self = !SHF && A.self != 0;               // (a run-time flag otherwise: the compiler versions the loops on it)
    const uint32_t total_units = __ldg(&A.offs[A.n_slabs]);
    const uint32_t n_batches = (total_units + JBATCH - 1) / JBATCH;
    const uint32_t r0 = join_cut(A.rowstart, A.nkeys, A.N, A.f0, A.fden), r1 = join_cut(A.rowstart, A.nkeys, A.N, A.f1, A.fden);   // this part's rows

    for (;;) {
        unsigned long long bi = 0;
        if (lane == 0) bi = atomicAdd(A.cursor, 1ull);
        bi = __shfl_sync(FULL, bi, 0);
        if (bi >= n_batches) break;
        const uint32_t u0 = (uint32_t)bi * JBATCH, u1 = min(total_units, u0 + JBATCH);
        // slab of the first unit: offs[lo] <= u0 < offs[hi] by a 32-ary search (offs is non-decreasing)
        uint32_t lo = 0, hi = A.n_slabs;
        while (hi - lo > 1) {
            const uint32_t step = (hi - lo + 32) / 33;
            const uint32_t pos = lo + (uint32_t)(lane + 1) * step;
            const bool le = pos < hi && __ldg(&A.offs[pos]) <= u0;
            const uint32_t k = (uint32_t)__popc(__ballot_sync(FULL, le));
            hi = min(hi, lo + (k + 1) * step);
            lo = lo + k * step;
        }
        uint32_t sl = lo;
        for (uint32_t u = u0; u < u1; u++) {
            for (;;) {                                   // skip slabs without units: first sl with offs[sl + 1] > u
                const uint32_t v = __ldg(&A.offs[min(sl + 1u + (uint32_t)lane, A.n_slabs)]);
                const unsigned m = __ballot_sync(FULL, v > u);
                if (m) { sl += (uint32_t)(__ffs(m) - 1); break; }
                sl += 32;
            }
            const uint32_t chunk = u - __ldg(&A.offs[sl]);
            const uint32_t i0 = sl * JROWS, i = i0 + (uint32_t)lane;
            const int first = (int)(max(i0, r0) - i0), last = (int)(min(min(A.N, i0 + (uint32_t)JROWS), r1) - i0) - 1;   // the slab's rows of this part
            const bool mine = lane >= first && lane <= last;
            const uint32_t x = mine ? __ldg(&A.rows[i]) : 0u;
            const uint32_t k = mine ? seed_key(x, ka) : 0xFFFFFFFFu;            // a row of another part (or a pad row) matches no column
            const uint32_t my_lo = mine ? __ldg(&A.colstart[k]) : 0u;           // this row's bucket on the column side
            const uint32_t my_hi = mine ? __ldg(&A.colstart[k + 1u]) : 0u;
            uint32_t run_lo = __shfl_sync(FULL, my_lo, first);
            const uint32_t run_hi = __shfl_sync(FULL, my_hi, last);
            if (self) run_lo = max(run_lo, i0 + (uint32_t)first + 1u);
            const uint32_t c0 = run_lo + chunk * (uint32_t)JUNIT, c1 = min(run_hi, c0 + (uint32_t)JUNIT);
            n_units++;
            for (uint32_t base = c0; base < c1; base += JCH) {
                const int ncols = (int)min((uint32_t)JCH, c1 - base);
                __syncwarp();                            // every lane is done with the previous sub-tile
                for (int t = 0; t * 32 < ncols + JPAD; t++) {
                    const uint32_t j = base + (uint32_t)(t * 32 + lane);
                    const bool real = t * 32 + lane < ncols;
                    const uint32_t y = real ? __ldg(&A.cols[j]) : 0u;
                    sb0[t * 32 + lane] = y;
                    sbP[t * 32 + lane] = y >> 2;
                    if constexpr (!SHF) sbM[t * 32 + lane] = y << 2;
                    sbK[t * 32 + lane] = real ? seed_key(y, kb) : 0xFFFFFFFEu;   // a pad column matches no row
                }
                __syncwarp();
#pragma unroll 1
                for (int q = first / RS; q * RS <= last; q++) {   // sub-slab q = rows q * RS .. + RS - 1 against their own column run
                    uint32_t s_lo = __shfl_sync(FULL, my_lo, max(q * RS, first));
                    const uint32_t s_hi = __shfl_sync(FULL, my_hi, min(q * RS + RS - 1, last));
                    const uint32_t xq = __shfl_sync(FULL, x, q * RS + r);
                    const uint32_t kq = __shfl_sync(FULL, k, q * RS + r);
                    const uint32_t iq = i0 + (uint32_t)(q * RS + r);
                    if (self) s_lo = max(s_lo, i0 + (uint32_t)max(q * RS, first) + 1u);
                    const uint32_t g_lo = max(s_lo, base), g_hi = min(s_hi, base + (uint32_t)ncols);
                    if (g_lo >= g_hi) continue;
                    const int gb = (int)(g_lo - base) & ~3, ge = (int)(g_hi - base);      // 16-byte aligned start
                    n_pairs += (unsigned long long)(ge - gb);
#pragma unroll 1
                    for (int g0 = gb; g0 < ge; g0 += 8 * STEP) {
                        uint32_t h = 0;
#pragma unroll 2
                        for (int st = 0; st < 8; st++) {
                            if (g0 + st * STEP < ge) {   // uniform across the warp
                                const int off = g0 + st * STEP + 4 * ph;
                                const uint4 B0 = *reinterpret_cast<const uint4*>(&sb0[off]);
                                const uint4 BP = *reinterpret_cast<const uint4*>(&sbP[off]);
                                const uint4 BM = SHF ? make_uint4(0u, 0u, 0u, 0u) : *reinterpret_cast<const uint4*>(&sbM[off]);
                                const uint4 BK = *reinterpret_cast<const uint4*>(&sbK[off]);
#pragma unroll
                                for (int kk = 0; kk < 4; kk++) {
                                    bool pass;
                                    if constexpr (T == 2) {
                                        pass = join2_quick<SHF>(xq, pick4(B0, kk), pick4(BP, kk), pick4(BM, kk), A.one, mone);
                                    } else {
                                        uint32_t w = quick3_marks(xq, pick4(B0, kk), pick4(BP, kk), pick4(BM, kk));
                                        w &= w * A.one + mone;   // drop the t lowest marks (IMAD keeps the -1 off the ALU pipe)
                                        w &= w * A.one + mone;
                                        w &= w * A.one + mone;
                                        pass = w == 0;
                                    }
                                    bool hit = pass && pick4(BK, kk) == kq;
                                    if (self) hit = hit && base + (uint32_t)(off + kk) > iq;
                                    h |= (hit ? 1u : 0u) << (st * 4 + kk);
                                }
                            }
                        }
                        if (__any_sync(FULL, h != 0)) {
                            n_cand += __popc(h);
                            join_push<T, STEP>(h, xq, sb0, g0 + 4 * ph, qn, q2n, c, out);
                        }
                    }
                }
            }
        }
    }
    join_drain<T>(c, out, qn, q2n, true);
    {                                                    // what is left in the scoring queues: fewer than 32 each
        const int n1 = T == 2 ? jfill(q2n, 0) : q2n, n2 = T == 2 ? jfill(q2n, 1) : 0;
        bool ok = false;
        uint32_t a = 0, b = 0;
        int d = 0;
        if (lane < n1) {
            const uint2 e = c.q2[lane];
            a = e.x; b = e.y; d = c.q2d[lane];
            ok = qgram_score_compact(a, b) >= A.T;
        }
        emit_warp(ok, a, b, d, out);
        if constexpr (T == 2) {                          // the far diagonals of the undecided
            ok = false;
            if (lane < n2) {
                const uint2 e = c.q2[JQ_FAR + lane];
                const uint8_t fd = c.q2d[JQ_FAR + lane];
                a = e.x; b = e.y; d = fd & 3;
                ok = (int)(fd >> 2) + qgram_score_far(a, b) >= A.T;
            }
            emit_warp(ok, a, b, d, out);
        }
    }
    if (A.stats) {
        for (int o = 16; o; o >>= 1) n_cand += __shfl_down_sync(FULL, n_cand, o);           // per-lane counts
        if (lane == 0) {                                                                  // the others are uniform per warp
            atomicAdd(&A.stats[0], n_units); atomicAdd(&A.stats[2], n_pairs * (unsigned long long)RS); atomicAdd(&A.stats[3], n_cand);
            atomicAdd(&A.stats[6], c.n_near); atomicAdd(&A.stats[7], c.n_owned);
            warp_exit_stats(A.stats, t_start);
        }
    }
}

}  // namespace bdg
