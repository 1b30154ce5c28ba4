// bdg_join3.cuh -- edge construction at t = 3 by sort-merge joins on multi-block seeds (bdg_seed3.cuh); sm_100a.
// Reference semantics: index.py:77-93 (candidate filter S >= T(3) = 4) + barcode_graph.py:233-249 (3-way edit-distance verify, emit).
//
// The machinery of the t = 2 join (bdg_join.cuh) with the t = 3 seed table: per condition the counting sort buckets both sides
// (join_hist_rank_kernel / join_scatter_rank_kernel, unchanged), join3_band_kernel counts the work units of every slab of 32
// rows, and one persistent join3_kernel launch walks them.  What differs per pair:
//   * quick test on the diagonals -2..2 (quick3_marks; the +-2 words are derived from the staged +-1 ones), three marks dropped;
//   * exact stage dist3_min (Myers' bit-vector pass; D <= 3 has no case analysis) and the hand-over walk seed3_first, in the
//     order the launch asks for (owner_first: the walk first, then the distance of the owned candidates only);
//   * the 6-mer score of the survivors through one scoring queue, full batches only, T = 4.
// The scheme is too large for constant memory next to the t = 2 one: the kernel reads the condition's two keys from its
// arguments and the hand-over tables from a device copy of the Seed3Scheme.
#pragma once
#include "bdg_join.cuh"
#include "bdg_seed3.cuh"

namespace bdg {

struct Join3Args {
    JoinArgs j;                     // rows / cols / bucket starts / unit offsets / cursor / stats / part cut, as at t = 2 (lut unused)
    SeedKey ka, kb;                 // the condition's row-side / column-side key
    const Seed3Scheme* scheme;      // device copy: hand-over tables
    int owner_first;                // 1: hand-over walk before the exact distance
};

// units of every slab of 32 rows (join_band_kernel with the key from the arguments)
__global__ void join3_band_kernel(const Join3Args A3, uint32_t* __restrict__ counts)
{
    const JoinArgs& A = A3.j;
    const uint32_t r0 = join_cut(A.rowstart, A.nkeys, A.N, A.f0, A.fden), r1 = join_cut(A.rowstart, A.nkeys, A.N, A.f1, A.fden);
    for (uint32_t s = blockIdx.x * blockDim.x + threadIdx.x; s <= A.n_slabs; s += gridDim.x * blockDim.x) {
        uint32_t cnt = 0;
        if (s < A.n_slabs) {
            const uint32_t i0 = max(s * JROWS, r0), i1 = min(min(A.N, s * JROWS + JROWS), r1);
            if (i0 < i1) {
                uint32_t lo = __ldg(&A.colstart[seed_key(__ldg(&A.rows[i0]), A3.ka)]);
                const uint32_t hi = __ldg(&A.colstart[seed_key(__ldg(&A.rows[i1 - 1u]), A3.ka) + 1u]);
                if (A.self) lo = max(lo, i0 + 1u);
                cnt = hi > lo ? (hi - lo + JUNIT - 1) / JUNIT : 0u;
            }
        }
        counts[s] = cnt;
    }
}

// Work estimate of the conditions c0 .. c1 - 1 of one block set over a sample (every stride-th barcode): table 0 holds the row
// key of the set (its first, symmetric, condition), table c - c0 the column key of condition c.
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

constexpr int J3Q2CAP = 64;        // scoring queue entries per warp

struct Join3Ctx {
    uint2* q;                      // candidates (x, y): row value, column value
    uint2* q2;                     // (a, b) with D <= 3 owned by this pass that still need the 6-mer score
    uint8_t* q2d;
    const Seed3Scheme* scheme;
    int lane, T, want0, want1, owner_first;
    unsigned long long n_d3, n_owned;
};

// exact stage on a batch of candidates (one per lane): D, hand-over walk, survivors into the scoring queue, full batches of that
// queue through the 6-mer score.  Not inlined, as at t = 2: one copy of the bit-vector pass, the walk and the score loop.
// Returns the queue fill | pairs with D <= 3 << 8 | pairs owned by this pass << 16.
__device__ __noinline__ uint32_t join3_process(uint2* q2, uint8_t* q2d, const Seed3Scheme* S, int want0, int want1, int owner_first, int T, const EdgeOut out,
                                               uint2 e, bool active, int n1)
{
    const int lane = threadIdx.x & 31;
    const uint32_t a = min(e.x, e.y), b = max(e.x, e.y);
    const int want = e.x > e.y ? want1 : want0;
    bool ok = active && a != b;
    int d = 4;
    uint32_t n_d3, n_own;
    if (owner_first) {
        if (ok) ok = seed3_first(*S, a, b) == want;      // emitted by the first (condition, orientation) the pair meets
        n_own = (uint32_t)__popc(__ballot_sync(FULL, ok));
        if (ok) { d = dist3_min(a, b); ok = d <= 3; }
        n_d3 = (uint32_t)__popc(__ballot_sync(FULL, ok));
    } else {
        if (ok) { d = dist3_min(a, b); ok = d <= 3; }
        n_d3 = (uint32_t)__popc(__ballot_sync(FULL, ok));
        if (ok) ok = seed3_first(*S, a, b) == want;
        n_own = (uint32_t)__popc(__ballot_sync(FULL, ok));
    }
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
    return (uint32_t)n1 | (n_d3 << 8) | (n_own << 16);
}

__device__ __forceinline__ void join3_drain(Join3Ctx& c, const EdgeOut& out, int& qn, int& q2n, bool all)
{
    __syncwarp();
    while (qn >= 32 || (all && qn > 0)) {
        const int take = min(qn, 32);
        qn -= take;
        const uint2 e = c.lane < take ? c.q[qn + c.lane] : make_uint2(0u, 0u);
        const uint32_t r = join3_process(c.q2, c.q2d, c.scheme, c.want0, c.want1, c.owner_first, c.T, out, e, c.lane < take, q2n);
        q2n = (int)(r & 255u);
        c.n_d3 += (r >> 8) & 255u;
        c.n_owned += r >> 16;
        __syncwarp();
    }
}

// append the hits of a group of 8 steps (join_push with the t = 3 exact stage)
template <int STEP>
__device__ __forceinline__ void join3_push(uint32_t h, uint32_t x, const uint32_t* sb0, int colbase, int& qn, int& q2n, Join3Ctx& c, const EdgeOut& out)
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
        int slot = qn + incl - cnt;
        while (h) {
            const int j = __ffs(h) - 1;
            h &= h - 1;
            c.q[slot++] = make_uint2(x, sb0[colbase + (j >> 2) * STEP + (j & 3)]);
        }
        qn += total;
        join3_drain(c, out, qn, q2n, false);
        return;
    }
    for (;;) {                                           // burst larger than the queue: one hit per lane and round
        const bool has = h != 0;
        const unsigned m = __ballot_sync(FULL, has);
        if (m == 0) break;
        if (has) {
            const int j = __ffs(h) - 1;
            h &= h - 1;
            c.q[qn + __popc(m & ((1u << c.lane) - 1u))] = make_uint2(x, sb0[colbase + (j >> 2) * STEP + (j & 3)]);
        }
        qn += __popc(m);
        join3_drain(c, out, qn, q2n, false);
    }
}

template <int RS>
__global__ void __launch_bounds__(ENT, 4) join3_kernel(const Join3Args A3, const EdgeOut out)
{
    constexpr int PH = 32 / RS;
    constexpr int STEP = 4 * PH;
    __shared__ __align__(16) uint32_t s_b[EW][4][JCH + JPAD];   // y, y >> 2, y << 2, key of the staged columns
    __shared__ uint2 s_q[EW][JQCAP];
    __shared__ uint2 s_q2[EW][J3Q2CAP];
    __shared__ uint8_t s_q2d[EW][J3Q2CAP];
    const JoinArgs& A = A3.j;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int r = lane & (RS - 1), ph = lane / RS;
    uint32_t* const sb0 = s_b[wid][0];
    uint32_t* const sbP = s_b[wid][1];
    uint32_t* const sbM = s_b[wid][2];
    uint32_t* const sbK = s_b[wid][3];
    Join3Ctx c;
    c.q = s_q[wid]; c.q2 = s_q2[wid]; c.q2d = s_q2d[wid]; c.scheme = A3.scheme; c.lane = lane; c.T = A.T;
    c.want0 = 2 * A.cond; c.want1 = 2 * A.cond + (A.self ? 0 : 1); c.owner_first = A3.owner_first; c.n_d3 = 0; c.n_owned = 0;
    int qn = 0, q2n = 0;
    const uint32_t mone = A.mone;
    const unsigned long long t_start = global_ns();
    unsigned long long n_units = 0, n_pairs = 0, n_cand = 0;
    const SeedKey& ka = A3.ka;
    const SeedKey& kb = A3.kb;
    const bool self = A.self != 0;
    const uint32_t total_units = __ldg(&A.offs[A.n_slabs]);
    const uint32_t n_batches = (total_units + JBATCH - 1) / JBATCH;
    const uint32_t r0 = join_cut(A.rowstart, A.nkeys, A.N, A.f0, A.fden), r1 = join_cut(A.rowstart, A.nkeys, A.N, A.f1, A.fden);

    for (;;) {
        unsigned long long bi = 0;
        if (lane == 0) bi = atomicAdd(A.cursor, 1ull);
        bi = __shfl_sync(FULL, bi, 0);
        if (bi >= n_batches) break;
        const uint32_t u0 = (uint32_t)bi * JBATCH, u1 = min(total_units, u0 + JBATCH);
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
            for (;;) {
                const uint32_t v = __ldg(&A.offs[min(sl + 1u + (uint32_t)lane, A.n_slabs)]);
                const unsigned m = __ballot_sync(FULL, v > u);
                if (m) { sl += (uint32_t)(__ffs(m) - 1); break; }
                sl += 32;
            }
            const uint32_t chunk = u - __ldg(&A.offs[sl]);
            const uint32_t i0 = sl * JROWS, i = i0 + (uint32_t)lane;
            const int first = (int)(max(i0, r0) - i0), last = (int)(min(min(A.N, i0 + (uint32_t)JROWS), r1) - i0) - 1;
            const bool mine = lane >= first && lane <= last;
            const uint32_t x = mine ? __ldg(&A.rows[i]) : 0u;
            const uint32_t k = mine ? seed_key(x, ka) : 0xFFFFFFFFu;
            const uint32_t my_lo = mine ? __ldg(&A.colstart[k]) : 0u;
            const uint32_t my_hi = mine ? __ldg(&A.colstart[k + 1u]) : 0u;
            uint32_t run_lo = __shfl_sync(FULL, my_lo, first);
            const uint32_t run_hi = __shfl_sync(FULL, my_hi, last);
            if (self) run_lo = max(run_lo, i0 + (uint32_t)first + 1u);
            const uint32_t c0 = run_lo + chunk * (uint32_t)JUNIT, c1 = min(run_hi, c0 + (uint32_t)JUNIT);
            n_units++;
            for (uint32_t base = c0; base < c1; base += JCH) {
                const int ncols = (int)min((uint32_t)JCH, c1 - base);
                __syncwarp();
                for (int t = 0; t * 32 < ncols + JPAD; t++) {
                    const uint32_t j = base + (uint32_t)(t * 32 + lane);
                    const bool real = t * 32 + lane < ncols;
                    const uint32_t y = real ? __ldg(&A.cols[j]) : 0u;
                    sb0[t * 32 + lane] = y;
                    sbP[t * 32 + lane] = y >> 2;
                    sbM[t * 32 + lane] = y << 2;
                    sbK[t * 32 + lane] = real ? seed_key(y, kb) : 0xFFFFFFFEu;
                }
                __syncwarp();
#pragma unroll 1
                for (int q = first / RS; q * RS <= last; q++) {
                    uint32_t s_lo = __shfl_sync(FULL, my_lo, max(q * RS, first));
                    const uint32_t s_hi = __shfl_sync(FULL, my_hi, min(q * RS + RS - 1, last));
                    const uint32_t xq = __shfl_sync(FULL, x, q * RS + r);
                    const uint32_t kq = __shfl_sync(FULL, k, q * RS + r);
                    const uint32_t iq = i0 + (uint32_t)(q * RS + r);
                    if (self) s_lo = max(s_lo, i0 + (uint32_t)max(q * RS, first) + 1u);
                    const uint32_t g_lo = max(s_lo, base), g_hi = min(s_hi, base + (uint32_t)ncols);
                    if (g_lo >= g_hi) continue;
                    const int gb = (int)(g_lo - base) & ~3, ge = (int)(g_hi - base);
                    n_pairs += (unsigned long long)(ge - gb);
#pragma unroll 1
                    for (int g0 = gb; g0 < ge; g0 += 8 * STEP) {
                        uint32_t h = 0;
#pragma unroll 2
                        for (int st = 0; st < 8; st++) {
                            if (g0 + st * STEP < ge) {
                                const int off = g0 + st * STEP + 4 * ph;
                                const uint4 B0 = *reinterpret_cast<const uint4*>(&sb0[off]);
                                const uint4 BP = *reinterpret_cast<const uint4*>(&sbP[off]);
                                const uint4 BM = *reinterpret_cast<const uint4*>(&sbM[off]);
                                const uint4 BK = *reinterpret_cast<const uint4*>(&sbK[off]);
#pragma unroll
                                for (int kk = 0; kk < 4; kk++) {
                                    uint32_t w = quick3_marks(xq, pick4(B0, kk), pick4(BP, kk), pick4(BM, kk));
                                    w &= w * A.one + mone;   // drop the three lowest marks
                                    w &= w * A.one + mone;
                                    w &= w * A.one + mone;
                                    bool hit = w == 0 && pick4(BK, kk) == kq;
                                    if (self) hit = hit && base + (uint32_t)(off + kk) > iq;
                                    h |= (hit ? 1u : 0u) << (st * 4 + kk);
                                }
                            }
                        }
                        if (__any_sync(FULL, h != 0)) {
                            n_cand += __popc(h);
                            join3_push<STEP>(h, xq, sb0, g0 + 4 * ph, qn, q2n, c, out);
                        }
                    }
                }
            }
        }
    }
    join3_drain(c, out, qn, q2n, true);
    {                                                    // what is left in the scoring queue: fewer than 32
        bool ok = false;
        uint32_t a = 0, b = 0;
        int d = 0;
        if (lane < q2n) {
            const uint2 e = c.q2[lane];
            a = e.x; b = e.y; d = c.q2d[lane];
            ok = qgram_score_compact(a, b) >= A.T;
        }
        emit_warp(ok, a, b, d, out);
    }
    if (A.stats) {
        for (int o = 16; o; o >>= 1) n_cand += __shfl_down_sync(FULL, n_cand, o);
        if (lane == 0) {
            atomicAdd(&A.stats[0], n_units); atomicAdd(&A.stats[2], n_pairs * (unsigned long long)RS); atomicAdd(&A.stats[3], n_cand);
            atomicAdd(&A.stats[6], c.n_d3); atomicAdd(&A.stats[7], c.n_owned);
            warp_exit_stats(A.stats, t_start);
        }
    }
}

}  // namespace bdg
