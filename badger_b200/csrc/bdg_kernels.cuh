// bdg_kernels.cuh -- hand-written CUDA kernels (sm_100a) for the barcode hot path.
//
// Kernel inventory (DESIGN.md has the roofline of each):
//   edges_kernel<MODE>   (bdg_edges.cuh) all-pairs edge construction over the sorted barcodes   INT-ALU bound
//   nearest_kernel       Q x W bounded plain edit distance, first minimum per query           INT-ALU bound
//   kmer_score_kernel    Q x W shared-6-mer product counts with per-position multiplicities   INT-ALU bound
//   kmer_unpack_kernel   packed position counts -> uint8[hits][11] (device form of a-5)        HBM bound
//   member_kernel        sorted-whitelist membership (smem pivots + L2-resident search)       HBM/L2 bound
//   pack16_kernel        16 ASCII bases -> 2-bit packed uint32 + validity                     HBM bound
//   tally_merge_kernel<B> merge path of the running distinct set and a batch's list / another set  HBM bound
//   lookup_assign32_kernel  per-read centre for rows outside a read map (smem pivots + search)  L2/HBM bound
//   pipe_probe_kernel    LOP3 / IMAD / POPC issue-rate probe for the integer roofline
//
// No tensor cores on purpose: nothing here is a dense contraction (BASELINE.json north_star).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "bdg_core.cuh"
#include "bdg_edges.cuh"

namespace bdg {

constexpr int NT = 256;            // threads per CTA

// ---------------------------------------------------------------------------------------------------
// nearest_kernel (a-7): every thread owns RA queries, the targets stream through shared memory in order,
// the t=2 prefilter guards the exact plain distance, and the running (distance, index) minimum lives in a
// register as one packed key so that "first strict minimum in caller order" is a plain unsigned min.
// gridDim.y splits the target list; the per-query keys are merged with atomicMin.
// ---------------------------------------------------------------------------------------------------
constexpr uint32_t NEAR_IDX_BITS = 28;
constexpr int NEAR_TB = 512;

template <bool SMALL>
__global__ void __launch_bounds__(NT, 2) nearest_kernel(const uint32_t* __restrict__ q, uint32_t Q,
                                                        const uint32_t* __restrict__ tg, uint32_t W, int max_d,
                                                        uint32_t w_per_block, uint32_t* __restrict__ keys)
{
    __shared__ __align__(16) uint32_t s_t[NEAR_TB];
    const int tid = threadIdx.x;
    uint32_t a[RA], best[RA];
#pragma unroll
    for (int r = 0; r < RA; r++) {
        const uint64_t idx = ((uint64_t)blockIdx.x * RA + r) * NT + tid;
        a[r] = idx < Q ? __ldg(&q[idx]) : 0u;
        best[r] = 0xFFFFFFFFu;
    }
    const uint32_t w_lo = blockIdx.y * w_per_block;
    const uint32_t w_hi = min(W, w_lo + w_per_block);
    for (uint32_t base = w_lo; base < w_hi; base += NEAR_TB) {
        __syncthreads();
        for (int x = tid; x < NEAR_TB; x += NT) s_t[x] = (base + x) < w_hi ? __ldg(&tg[base + x]) : 0u;
        __syncthreads();
        const int n = min((uint32_t)NEAR_TB, w_hi - base);
        for (int x = 0; x < n; x++) {
            const uint32_t b = s_t[x];
            const uint32_t bR = b >> 2, bL = b << 2;
#pragma unroll
            for (int r = 0; r < RA; r++) {
                int d;
                if (SMALL) {
                    const uint32_t x0 = a[r] ^ b, x1 = a[r] ^ bR, x2 = a[r] ^ bL;
                    const uint32_t m = ((x0 - F10_ONES) & ~x0) | ((x1 - F10_ONES) & ~x1) | ((x2 - F10_ONES) & ~x2);
                    if (!(m & F10_HIGH)) continue;
                    d = dist_small(a[r], b, true);
                } else {
                    d = myers3(a[r], b).full;
                }
                if (d <= max_d) best[r] = min(best[r], ((uint32_t)d << NEAR_IDX_BITS) | (base + x));
            }
        }
    }
#pragma unroll
    for (int r = 0; r < RA; r++) {
        const uint64_t idx = ((uint64_t)blockIdx.x * RA + r) * NT + tid;
        if (idx < Q && best[r] != 0xFFFFFFFFu) atomicMin(&keys[idx], best[r]);
    }
}

__global__ void nearest_finish_kernel(const uint32_t* __restrict__ keys, uint32_t Q, int32_t* __restrict__ argmin,
                                      uint8_t* __restrict__ dist)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= Q) return;
    const uint32_t k = keys[i];
    if (k == 0xFFFFFFFFu) { argmin[i] = -1; dist[i] = 255; }
    else { argmin[i] = (int32_t)(k & ((1u << NEAR_IDX_BITS) - 1u)); dist[i] = (uint8_t)(k >> NEAR_IDX_BITS); }
}

// ---------------------------------------------------------------------------------------------------
// Posting-list form of the same operator (the reference's own data structure, kmer_indexer.py:29-32 / index.py:29-41, on the
// device): the known strings' 6-mers as 4096 buckets of string ids (a 6-mer that occurs twice in a string is listed once).
// A query walks the buckets of its own 6-mers: work = sum of <= 11 bucket sizes (~3 % of W for random strings) instead of W.
//   kidx_hist_kernel / kidx_scatter_kernel   counting sort of the (6-mer, id) postings (one digit of 12 bits)
//   kmer_post_kernel                          one CTA per (query, query position p): skipped when the 6-mer at p already occurred
//                                             at an earlier position of the query; else every id of the bucket gets the exact
//                                             score, and is emitted from THIS bucket iff p is the first query position whose
//                                             6-mer occurs in the entry (so every hit is emitted exactly once).
// ---------------------------------------------------------------------------------------------------
__global__ void kidx_hist_kernel(const uint32_t* __restrict__ wl, uint32_t W, uint32_t* __restrict__ hist)
{
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < W; i += gridDim.x * blockDim.x) {
        const uint32_t w = __ldg(&wl[i]);
        for (int p = 0; p <= 10; p++)
            if (!kmer_seen_before(w, p)) atomicAdd(&hist[(w >> (2 * p)) & 0xFFFu], 1u);
    }
}

__global__ void kidx_scatter_kernel(const uint32_t* __restrict__ wl, uint32_t W, const uint32_t* __restrict__ start, uint32_t* __restrict__ fill,
                                    uint32_t* __restrict__ post)
{
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < W; i += gridDim.x * blockDim.x) {
        const uint32_t w = __ldg(&wl[i]);
        for (int p = 0; p <= 10; p++) {
            if (kmer_seen_before(w, p)) continue;
            const uint32_t k = (w >> (2 * p)) & 0xFFFu;
            post[__ldg(&start[k]) + atomicAdd(&fill[k], 1u)] = i;
        }
    }
}

__global__ void __launch_bounds__(NT) kmer_post_kernel(const uint32_t* __restrict__ q, uint32_t Q, const uint32_t* __restrict__ wl,
                                                       const uint32_t* __restrict__ start, const uint32_t* __restrict__ post, int min_kmers,
                                                       unsigned long long cap, uint32_t* __restrict__ hit_q, uint32_t* __restrict__ hit_w,
                                                       uint8_t* __restrict__ cnt, unsigned long long* __restrict__ mult,
                                                       unsigned long long* __restrict__ total)
{
    const int lane = threadIdx.x & 31;
    for (uint64_t item = blockIdx.x; item < (uint64_t)Q * 11; item += gridDim.x) {
        const uint32_t qi = (uint32_t)(item / 11);
        const int p = (int)(item % 11);
        const uint32_t a = __ldg(&q[qi]);
        if (kmer_seen_before(a, p)) continue;                         // that bucket was walked for the earlier position
        const uint32_t k = (a >> (2 * p)) & 0xFFFu;
        const uint32_t lo = __ldg(&start[k]), hi = __ldg(&start[k + 1]);
        for (uint32_t base = lo; base < hi; base += NT) {             // whole warps stay in the loop together
            const uint32_t j = base + threadIdx.x;
            bool ok = false;
            uint32_t wi = 0, b = 0;
            int s = 0;
            if (j < hi) {
                wi = __ldg(&post[j]);
                b = __ldg(&wl[wi]);
                uint32_t marks = 0;
                s = qgram_score_marks(a, b, &marks);
                ok = s >= min_kmers && (marks & ((1u << (2 * p)) - 1u)) == 0;      // no earlier query position has a 6-mer of this entry
            }
            const unsigned m = __ballot_sync(0xffffffffu, ok);
            if (m == 0) continue;
            unsigned long long at = 0;
            const int leader = __ffs(m) - 1;
            if (lane == leader) at = atomicAdd(total, (unsigned long long)__popc(m));
            at = __shfl_sync(0xffffffffu, at, leader);
            if (ok) {
                const unsigned long long pos = at + __popc(m & ((1u << lane) - 1u));
                if (pos < cap) {
                    uint64_t mu;
                    qgram_score(a, b, &mu);
                    hit_q[pos] = qi;
                    hit_w[pos] = wi;
                    cnt[pos] = (uint8_t)s;
                    mult[pos] = mu;
                }
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------------
// kmer_score_kernel (a-5), brute-force form (kept for small string sets): thread per whitelist entry, queries broadcast from
// shared memory; exact S with
// per-position multiplicities; hits appended through a warp-aggregated cursor.
// ---------------------------------------------------------------------------------------------------
constexpr int KS_QB = 256;

__global__ void __launch_bounds__(NT) kmer_score_kernel(const uint32_t* __restrict__ q, uint32_t Q,
                                                        const uint32_t* __restrict__ wl, uint32_t W, int min_kmers,
                                                        unsigned long long cap, uint32_t* __restrict__ hit_q,
                                                        uint32_t* __restrict__ hit_w, uint8_t* __restrict__ cnt,
                                                        unsigned long long* __restrict__ mult,
                                                        unsigned long long* __restrict__ total)
{
    __shared__ uint32_t s_q[KS_QB];
    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const uint64_t wi = (uint64_t)blockIdx.x * NT + tid;
    const uint32_t b = wi < W ? __ldg(&wl[wi]) : 0u;
    const uint32_t q_lo = blockIdx.y * KS_QB;
    const int nq = min((uint32_t)KS_QB, Q - q_lo);
    for (int x = tid; x < nq; x += NT) s_q[x] = __ldg(&q[q_lo + x]);
    __syncthreads();
    for (int x = 0; x < nq; x++) {
        const uint32_t a = s_q[x];
        const int s = wi < W ? qgram_score(a, b) : 0;
        const bool ok = wi < W && s >= min_kmers && s > 0;
        const unsigned m = __ballot_sync(0xffffffffu, ok);
        if (m == 0) continue;
        unsigned long long base = 0;
        const int leader = __ffs(m) - 1;
        if (lane == leader) base = atomicAdd(total, (unsigned long long)__popc(m));
        base = __shfl_sync(0xffffffffu, base, leader);
        if (ok) {
            const unsigned long long pos = base + __popc(m & ((1u << lane) - 1u));
            if (pos < cap) {
                uint64_t mu;
                qgram_score(a, b, &mu);
                hit_q[pos] = q_lo + x;
                hit_w[pos] = (uint32_t)wi;
                cnt[pos] = (uint8_t)s;
                mult[pos] = mu;
            }
        }
    }
}

// kmer_unpack_kernel (a-5, device form): the 4-bit position counts of n hits (mult, nibble p = query position p) as uint8[n][11],
// the layout of the host operator's result.  One thread per output byte, so the writes are coalesced.
__global__ void kmer_unpack_kernel(const unsigned long long* __restrict__ mult, uint64_t n, uint8_t* __restrict__ pos)
{
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n * 11; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t h = i / 11;
        pos[i] = (uint8_t)((__ldg(&mult[h]) >> (4 * (i - h * 11))) & 15u);
    }
}

// ---------------------------------------------------------------------------------------------------
// member_kernel (a-6): 1024 evenly spaced pivots of the sorted whitelist in shared memory give the first
// ten levels of the search; the remaining levels touch a window of W/1024 entries (L2-resident: the 3 M
// whitelist is 12 MB).  4 B in + 1 B out per query.
// ---------------------------------------------------------------------------------------------------
constexpr int MEM_PIV = 1024;

__global__ void __launch_bounds__(NT) member_kernel(const uint32_t* __restrict__ wl, uint32_t W,
                                                    const uint32_t* __restrict__ q, uint32_t Q, uint8_t* __restrict__ hit)
{
    __shared__ uint32_t s_p[MEM_PIV];
    const uint64_t step = ((uint64_t)W + MEM_PIV - 1) / MEM_PIV;   // pivot p = wl[min(W-1, p*step)]
    for (int p = threadIdx.x; p < MEM_PIV; p += NT) {
        const uint64_t i = (uint64_t)p * step;
        s_p[p] = __ldg(&wl[i < W ? i : W - 1]);
    }
    __syncthreads();
    for (uint64_t i = (uint64_t)blockIdx.x * NT + threadIdx.x; i < Q; i += (uint64_t)gridDim.x * NT) {
        const uint32_t v = __ldg(&q[i]);
        int lo = 0, hi = MEM_PIV;   // largest pivot index with s_p[p] <= v (or 0)
#pragma unroll
        for (int it = 0; it < 10; it++) {
            const int mid = (lo + hi) >> 1;
            if (s_p[mid] <= v) lo = mid; else hi = mid;
        }
        uint64_t l = (uint64_t)lo * step, h = min((uint64_t)W, l + step);   // candidates in [l, h)
        if (l >= W) { l = W - 1; h = W; }
        while (l < h) {
            const uint64_t mid = (l + h) >> 1;
            if (__ldg(&wl[mid]) < v) l = mid + 1; else h = mid;
        }
        hit[i] = (l < W && __ldg(&wl[l]) == v) ? 1 : 0;
    }
}

// ---------------------------------------------------------------------------------------------------
// pack16_kernel (a-1): one 128-bit load per read, 16 B in + 5 B out.  code = ((c>>1) ^ (c>>2)) & 3 maps
// A,C,G,T -> 0,1,2,3; validity is an exact match against the four upper-case letters.
// ---------------------------------------------------------------------------------------------------
// four characters at once (SWAR): x = codes in the low two bits of every byte; a multiply gathers them into one
// byte (c0 | c1<<2 | c2<<4 | c3<<6 lands in bits 24..31, no carries: every partial product has its own 2-bit slot);
// validity = the four letters those codes stand for, looked up with byte permutes (the selector nibbles 0 and 2 of
// x and of x >> 16 are the codes, nibbles 1 and 3 are zero), equal the input word.
__device__ __forceinline__ void pack4(uint32_t wrd, int base_pos, uint32_t& r, bool& ok)
{
    const uint32_t x = ((wrd >> 1) ^ (wrd >> 2)) & 0x03030303u;
    r |= ((x * 0x01041040u) >> 24) << (2 * base_pos);
    const uint32_t e01 = __byte_perm(0x54474341u /* "ACGT" */, 0u, x);          // bytes 0, 2 = letters of characters 0, 1
    const uint32_t e23 = __byte_perm(0x54474341u, 0u, x >> 16);                 // bytes 0, 2 = letters of characters 2, 3
    ok = ok && (__byte_perm(e01, e23, 0x6420u) == wrd);
}

__global__ void __launch_bounds__(NT) pack16_kernel(const uint4* __restrict__ seqs, uint64_t R, uint32_t* __restrict__ out,
                                                    uint8_t* __restrict__ valid)
{
    // four independent 128-bit loads in flight per thread (one per 256-read row of a 1024-read block)
    constexpr int U = 4;
    for (uint64_t base = (uint64_t)blockIdx.x * NT * U; base < R; base += (uint64_t)gridDim.x * NT * U) {
        uint4 v[U];
#pragma unroll
        for (int u = 0; u < U; u++) {
            const uint64_t i = base + (uint64_t)u * NT + threadIdx.x;
            v[u] = i < R ? __ldg(&seqs[i]) : make_uint4(0u, 0u, 0u, 0u);
        }
#pragma unroll
        for (int u = 0; u < U; u++) {
            const uint64_t i = base + (uint64_t)u * NT + threadIdx.x;
            if (i < R) {
                uint32_t r = 0;
                bool ok = true;
                pack4(v[u].x, 0, r, ok); pack4(v[u].y, 4, r, ok); pack4(v[u].z, 8, r, ok); pack4(v[u].w, 12, r, ok);
                out[i] = r;
                valid[i] = ok ? 1 : 0;
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------------
// pipe_probe_kernel: 64 independent instructions per loop trip (8 chains x 8), inline PTX so that ptxas
// keeps the opcode.  kind 0 LOP3, 1 IMAD, 2 alternating LOP3/IMAD, 3 POPC(+LOP3 to keep chains alive).
// ---------------------------------------------------------------------------------------------------
template <int KIND>
__global__ void __launch_bounds__(NT) pipe_probe_kernel(int iters, uint32_t* __restrict__ sink)
{
    uint32_t v[8];
#pragma unroll
    for (int i = 0; i < 8; i++) v[i] = threadIdx.x * 2654435761u + i * 40503u + blockIdx.x;
    uint32_t c = sink[0] | 0x9E3779B9u, m = sink[1] | 5u;
    for (int it = 0; it < iters; it++) {
#pragma unroll
        for (int u = 0; u < 8; u++) {
#pragma unroll
            for (int i = 0; i < 8; i++) {
                if (KIND == 0 || (KIND == 2 && (u & 1) == 0))
                    asm volatile("lop3.b32 %0, %0, %1, %2, 0x96;" : "+r"(v[i]) : "r"(c), "r"(m));
                else if (KIND == 1 || KIND == 2)
                    asm volatile("mad.lo.u32 %0, %0, %1, %2;" : "+r"(v[i]) : "r"(m), "r"(c));
                else
                    asm volatile("popc.b32 %0, %0;" : "+r"(v[i]));
            }
        }
    }
    uint32_t s = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) s ^= v[i];
    if (s == 0x12345678u) sink[2] = s;   // practically never; keeps the chains live
}

// ---------------------------------------------------------------------------------------------------
// Dedup + count in FIRST-SEEN order (a-2, reference barcode_graph.py:192-204: `counts[rank] += 1`, dict order =
// order of first sighting).  The reads are radix-sorted by (key) with their read index as payload (stable: equal
// keys keep ascending indices, so the head of a run is the first sighting), then:
//   dedup_heads_kernel    head flags of the runs of equal keys
//   dedup_runs_kernel     per run (numbered by the exclusive scan of the heads): key, first read index, start
//   dedup_finish_kernel   after the runs are sorted by first read index: first-seen position of every run,
//                         distinct[] / counts[] in that order
//   dedup_scatter_kernel  read -> first-seen position of its barcode
// HBM bound: 4 B in per read for the flags, 4+4 B out for the per-read map; the sorts are cub (library, 2 passes).
// ---------------------------------------------------------------------------------------------------
__global__ void iota_kernel(uint32_t* __restrict__ v, uint32_t n)
{
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) v[i] = i;
}

__global__ void dedup_heads_kernel(const uint32_t* __restrict__ sk, uint32_t n, uint32_t* __restrict__ head)
{
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
        head[i] = (i == 0 || __ldg(&sk[i]) != __ldg(&sk[i - 1])) ? 1u : 0u;
}

// run_of[i] = inclusive scan of head - 1
__global__ void dedup_runs_kernel(const uint32_t* __restrict__ sk, const uint32_t* __restrict__ si, const uint32_t* __restrict__ head,
                                  const uint32_t* __restrict__ scan_incl, uint32_t n, uint32_t* __restrict__ run_key,
                                  uint32_t* __restrict__ run_first, uint32_t* __restrict__ run_start)
{
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        if (__ldg(&head[i])) {
            const uint32_t r = __ldg(&scan_incl[i]) - 1u;
            run_key[r] = __ldg(&sk[i]);
            run_first[r] = __ldg(&si[i]);
            run_start[r] = i;
        }
    }
}

// order[pos] = run with the pos-th smallest first read index
__global__ void dedup_finish_kernel(const uint32_t* __restrict__ order, const uint32_t* __restrict__ run_key,
                                    const uint32_t* __restrict__ run_start, uint32_t n_runs, uint32_t n_reads,
                                    uint32_t* __restrict__ distinct, uint32_t* __restrict__ counts, uint32_t* __restrict__ pos_of_run)
{
    for (uint32_t p = blockIdx.x * blockDim.x + threadIdx.x; p < n_runs; p += gridDim.x * blockDim.x) {
        const uint32_t r = __ldg(&order[p]);
        const uint32_t s0 = __ldg(&run_start[r]);
        const uint32_t s1 = r + 1 < n_runs ? __ldg(&run_start[r + 1]) : n_reads;
        distinct[p] = __ldg(&run_key[r]);
        counts[p] = s1 - s0;
        pos_of_run[r] = p;
    }
}

__global__ void dedup_scatter_kernel(const uint32_t* __restrict__ si, const uint32_t* __restrict__ scan_incl,
                                     const uint32_t* __restrict__ pos_of_run, uint32_t n, uint32_t* __restrict__ read_to_distinct)
{
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
        read_to_distinct[__ldg(&si[i])] = __ldg(&pos_of_run[__ldg(&scan_incl[i]) - 1u]);
}

// ---------------------------------------------------------------------------------------------------
// Merge of the dedup results of P parts (one process per GPU, bdg_dev_dedup_merge): every part brings its distinct barcodes
// ascending, their counts and their local first-seen positions.  The first sighting of a barcode over all parts is the
// smallest (part, local position), one 32-bit key: offset of the part (the sizes of the parts before it) + position.
//   merge_gather_kernel   the P lists (part p at starts[p], offs[p+1]-offs[p] entries) -> one concatenation with the first
//                         key of every entry; the entries of part `mine` are compared with the caller's own list
//   (radix sort by barcode, dedup_heads_kernel, inclusive scan: runs of equal barcodes, at most P entries each)
//   merge_runs_kernel     per run: barcode, summed count, smallest first key; for the entries of part `mine`, the run
//   (radix sort of the runs by first key: the global first-seen order)
//   merge_finish_kernel   distinct / counts in first-seen order and the first-seen position of every run
//   merge_local_kernel    local first-seen position of part `mine` -> global first-seen position
//   merge_remap_kernel    the read -> barcode map of part `mine` rewritten through that table
// ---------------------------------------------------------------------------------------------------
__global__ void merge_gather_kernel(const uint32_t* __restrict__ keys, const uint32_t* __restrict__ counts, const uint32_t* __restrict__ first,
                                    const uint64_t* __restrict__ starts, const uint32_t* __restrict__ offs, uint32_t P, uint32_t total,
                                    uint32_t mine, const uint32_t* __restrict__ own_sorted, uint32_t* __restrict__ out_key,
                                    uint32_t* __restrict__ out_idx, uint32_t* __restrict__ out_count, uint32_t* __restrict__ out_first,
                                    unsigned int* __restrict__ bad)
{
    for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; j < total; j += gridDim.x * blockDim.x) {
        uint32_t lo = 0, hi = P;                               // part p with offs[p] <= j < offs[p + 1]
        while (hi - lo > 1) {
            const uint32_t mid = (lo + hi) >> 1;
            if (__ldg(&offs[mid]) <= j) lo = mid; else hi = mid;
        }
        const uint32_t q = j - __ldg(&offs[lo]);
        const uint64_t src = __ldg(&starts[lo]) + q;
        const uint32_t k = __ldg(&keys[src]);
        out_key[j] = k;
        out_idx[j] = j;
        out_count[j] = __ldg(&counts[src]);
        out_first[j] = __ldg(&offs[lo]) + __ldg(&first[src]);
        if (lo == mine && __ldg(&own_sorted[q]) != k) *bad = 1u;
    }
}

__global__ void merge_runs_kernel(const uint32_t* __restrict__ sk, const uint32_t* __restrict__ si, const uint32_t* __restrict__ head,
                                  const uint32_t* __restrict__ scan_incl, uint32_t n, const uint32_t* __restrict__ count,
                                  const uint32_t* __restrict__ first, uint32_t mine_off, uint32_t mine_n, uint32_t* __restrict__ run_key,
                                  uint32_t* __restrict__ run_count, uint32_t* __restrict__ run_first, uint32_t* __restrict__ mine_run)
{
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        if (!__ldg(&head[i])) continue;
        const uint32_t r = __ldg(&scan_incl[i]) - 1u;
        uint32_t c = 0, f = 0xFFFFFFFFu;
        for (uint32_t j = i; j < n && (j == i || !__ldg(&head[j])); j++) {
            const uint32_t e = __ldg(&si[j]);
            c += __ldg(&count[e]);
            f = min(f, __ldg(&first[e]));
            if (e - mine_off < mine_n) mine_run[e - mine_off] = r;   // (unsigned: e < mine_off wraps above mine_n)
        }
        run_key[r] = __ldg(&sk[i]);
        run_count[r] = c;
        run_first[r] = f;
    }
}

// order[pos] = run with the pos-th smallest first key
__global__ void merge_finish_kernel(const uint32_t* __restrict__ order, const uint32_t* __restrict__ run_key, const uint32_t* __restrict__ run_count,
                                    uint32_t n_runs, uint32_t* __restrict__ distinct, uint32_t* __restrict__ counts, uint32_t* __restrict__ pos_of_run)
{
    for (uint32_t p = blockIdx.x * blockDim.x + threadIdx.x; p < n_runs; p += gridDim.x * blockDim.x) {
        const uint32_t r = __ldg(&order[p]);
        distinct[p] = __ldg(&run_key[r]);
        counts[p] = __ldg(&run_count[r]);
        pos_of_run[r] = p;
    }
}

// own_sorted_pos[q] = ascending position of the part's q-th barcode in first-seen order (its own list)
__global__ void merge_local_kernel(const uint32_t* __restrict__ own_sorted_pos, const uint32_t* __restrict__ mine_run,
                                   const uint32_t* __restrict__ pos_of_run, uint32_t n, uint32_t* __restrict__ global_pos)
{
    for (uint32_t q = blockIdx.x * blockDim.x + threadIdx.x; q < n; q += gridDim.x * blockDim.x)
        global_pos[q] = __ldg(&pos_of_run[__ldg(&mine_run[__ldg(&own_sorted_pos[q])])]);
}

__global__ void merge_remap_kernel(uint32_t* __restrict__ read_to_distinct, uint32_t n, const uint32_t* __restrict__ global_pos)
{
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
        read_to_distinct[i] = __ldg(&global_pos[read_to_distinct[i]]);
}

// ---------------------------------------------------------------------------------------------------
// Tally of reads that arrive in batches (bdg_tally_*): the running distinct set is ascending by barcode with a 64-bit count and a
// 64-bit first-sighting key per barcode; every batch is deduplicated as above and its ascending list is merged into the set.
//   tally_merge_kernel   merge path of the set A (na) and the batch B (nb): CTA k owns outputs [k*TALLY_TILE, (k+1)*TALLY_TILE),
//                        finds where that stretch of the merged order starts and ends in A and B (two binary searches along the
//                        cross diagonals), stages both key ranges in shared memory, and every thread merges TALLY_ITEMS outputs
//                        from its own diagonal.  Ties take A first, so a barcode the set already holds is followed directly by
//                        the batch's entry of it, which is flagged as no head.  B is read through an accessor (template
//                        parameter): TallyBatchSide, a batch's dedup output, or TallySetSide, the set of another tally
//                        (bdg_dev_tally_merge_parts folds the sets of P ranks one by one; each set is distinct, so a head is still
//                        followed by at most one non-head).
//   (inclusive scan of the heads: the position of every run in the new set)
//   tally_compact_kernel one entry per head, the count of a following non-head added in; counts of 2^32 or more are flagged
//   (radix sort of the set by first-sighting key at tally_finish: the global first-seen order)
//   tally_finish_kernel  distinct / counts (uint32) / first-seen -> ascending position, the read-map arrays of a dedup call
//   tally_part_check_kernel  the checks of bdg_dev_tally_merge_parts on one part before the fold
// HBM bound: 20 B in and 24 B out per merged entry, then 24 B in and 20 B out per entry of the new set.
// ---------------------------------------------------------------------------------------------------
constexpr int TALLY_ITEMS = 8;
constexpr int TALLY_TILE = NT * TALLY_ITEMS;

// B of the merge: n entries, key[j] the j-th smallest barcode; at(j) locates entry j in the arrays x and y, count(at(j)) and
// first(at(j)) are its count and first-sighting key.  The kernel takes key, x, y, n and first_off as separate parameters, in the
// batch form's former order and types, so the batch form compiles as before.
// A batch's dedup output: y[j] is run j's first-seen position in the batch, x the counts in first-seen order, first_off the rows
// added before the batch.
struct TallyBatchSide {
    using X = uint32_t;
    using Y = uint32_t;
    const uint32_t* key;
    const X* x;
    const Y* y;
    uint64_t n;
    unsigned long long first_off;
    __device__ __forceinline__ uint32_t at(uint64_t j) const { return __ldg(&y[j]); }
    __device__ __forceinline__ unsigned long long count(uint32_t p) const { return __ldg(&x[p]); }
    __device__ __forceinline__ unsigned long long first(uint32_t p) const { return first_off + p; }
};

// The running set of another tally: 64-bit counts x, 64-bit first-sighting keys y, shifted by first_off (the rows of the parts
// before it).
struct TallySetSide {
    using X = unsigned long long;
    using Y = unsigned long long;
    const uint32_t* key;
    const X* x;
    const Y* y;
    uint64_t n;
    unsigned long long first_off;
    __device__ __forceinline__ uint64_t at(uint64_t j) const { return j; }
    __device__ __forceinline__ unsigned long long count(uint64_t j) const { return __ldg(&x[j]); }
    __device__ __forceinline__ unsigned long long first(uint64_t j) const { return first_off + __ldg(&y[j]); }
};

// number of A entries among the first d outputs of the merge (ties: A first)
template <typename GetA, typename GetB>
__device__ __forceinline__ uint64_t merge_path_split(uint64_t d, uint64_t na, uint64_t nb, GetA a, GetB b)
{
    uint64_t lo = d > nb ? d - nb : 0, hi = d < na ? d : na;
    while (lo < hi) {
        const uint64_t mid = (lo + hi) >> 1;
        if (a(mid) <= b(d - 1 - mid)) lo = mid + 1; else hi = mid;
    }
    return lo;
}

template <typename BSide>
__global__ void __launch_bounds__(NT) tally_merge_kernel(const uint32_t* __restrict__ a_key, const unsigned long long* __restrict__ a_cnt,
                                                         const unsigned long long* __restrict__ a_first, uint64_t na,
                                                         const uint32_t* __restrict__ b_key, const typename BSide::X* __restrict__ b_x,
                                                         const typename BSide::Y* __restrict__ b_y, uint64_t nb, unsigned long long first_off,
                                                         uint32_t* __restrict__ m_key, unsigned long long* __restrict__ m_cnt,
                                                         unsigned long long* __restrict__ m_first, uint32_t* __restrict__ m_head)
{
    __shared__ uint32_t s_key[TALLY_TILE];
    __shared__ uint64_t s_split[2];
    const BSide b{b_key, b_x, b_y, nb, first_off};
    const uint64_t M = na + nb;
    const uint64_t d0 = (uint64_t)blockIdx.x * TALLY_TILE, d1 = min(M, d0 + TALLY_TILE);
    auto ga = [&](uint64_t i) { return __ldg(&a_key[i]); };
    auto gb = [&](uint64_t j) { return __ldg(&b_key[j]); };
    if (threadIdx.x < 2) s_split[threadIdx.x] = merge_path_split(threadIdx.x ? d1 : d0, na, nb, ga, gb);
    __syncthreads();
    const uint64_t a0 = s_split[0], a1 = s_split[1], b0 = d0 - a0, b1 = d1 - a1;
    const uint32_t la = (uint32_t)(a1 - a0), lb = (uint32_t)(b1 - b0);     // la + lb = d1 - d0 <= TALLY_TILE
    for (uint32_t k = threadIdx.x; k < la + lb; k += NT) s_key[k] = k < la ? ga(a0 + k) : gb(b0 + k - la);
    __syncthreads();
    const uint32_t* sa = s_key;
    const uint32_t* sb = s_key + la;
    const uint32_t dt = min((uint32_t)threadIdx.x * TALLY_ITEMS, la + lb);
    uint32_t i = (uint32_t)merge_path_split(dt, la, lb, [&](uint64_t x) { return sa[x]; }, [&](uint64_t y) { return sb[y]; });
    uint32_t j = dt - i;
    // the A entry right before this thread's first output (the one a batch entry of the same barcode follows)
    const bool have_prev = a0 + i > 0;
    uint32_t prev_a = have_prev ? (i > 0 ? sa[i - 1] : ga(a0 - 1)) : 0u;
    const uint32_t end = min(dt + TALLY_ITEMS, la + lb);
    bool any_a = have_prev;
    for (uint32_t o = dt; o < end; o++) {
        const uint64_t g = d0 + o;
        if (j >= lb || (i < la && sa[i] <= sb[j])) {
            const uint64_t ai = a0 + i;
            m_key[g] = sa[i];
            m_cnt[g] = __ldg(&a_cnt[ai]);
            m_first[g] = __ldg(&a_first[ai]);
            m_head[g] = 1u;
            prev_a = sa[i];
            any_a = true;
            i++;
        } else {
            const uint32_t k = sb[j];
            const auto p = b.at(b0 + j);
            m_key[g] = k;
            m_cnt[g] = b.count(p);
            m_first[g] = b.first(p);
            m_head[g] = (any_a && prev_a == k) ? 0u : 1u;
            j++;
        }
    }
}

// scan_incl[o] - 1 = position of head o in the new set; a non-head is always the entry right after its head
__global__ void tally_compact_kernel(const uint32_t* __restrict__ m_key, const unsigned long long* __restrict__ m_cnt,
                                     const unsigned long long* __restrict__ m_first, const uint32_t* __restrict__ m_head,
                                     const uint32_t* __restrict__ scan_incl, uint64_t M, uint32_t* __restrict__ key,
                                     unsigned long long* __restrict__ cnt, unsigned long long* __restrict__ first, unsigned int* __restrict__ over)
{
    for (uint64_t o = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; o < M; o += (uint64_t)gridDim.x * blockDim.x) {
        if (!__ldg(&m_head[o])) continue;
        const uint32_t r = __ldg(&scan_incl[o]) - 1u;
        unsigned long long c = __ldg(&m_cnt[o]), f = __ldg(&m_first[o]);
        if (o + 1 < M && !__ldg(&m_head[o + 1])) {
            c += __ldg(&m_cnt[o + 1]);
            f = min(f, __ldg(&m_first[o + 1]));
        }
        key[r] = __ldg(&m_key[o]);
        cnt[r] = c;
        first[r] = f;
        if (c >> 32) *over = 1u;
    }
}

// One part of bdg_dev_tally_merge_parts: bit 1 of *bad when its keys are not strictly ascending, bit 4 when a shifted first key is
// not below the total rows; when own_key is given (the caller's own part), bit 2 when an entry differs from the handle's set.
__global__ void tally_part_check_kernel(const TallySetSide b, unsigned long long rows, const uint32_t* __restrict__ own_key,
                                        const unsigned long long* __restrict__ own_cnt, const unsigned long long* __restrict__ own_first,
                                        unsigned int* __restrict__ bad)
{
    unsigned int f = 0;
    for (uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; j < b.n; j += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t k = __ldg(&b.key[j]);
        const unsigned long long c = b.count(j), first = b.first(j);
        if (j > 0 && __ldg(&b.key[j - 1]) >= k) f |= 1u;
        if (first >= rows || first < b.first_off) f |= 4u;
        if (own_key && (__ldg(&own_key[j]) != k || __ldg(&own_cnt[j]) != c || __ldg(&own_first[j]) + b.first_off != first)) f |= 2u;
    }
    if (f) atomicOr(bad, f);
}

// order[p] = ascending position of the barcode with the p-th smallest first-sighting key
__global__ void tally_finish_kernel(const uint32_t* __restrict__ order, const uint32_t* __restrict__ key, const unsigned long long* __restrict__ cnt,
                                    uint32_t n, uint32_t* __restrict__ distinct, uint32_t* __restrict__ counts, uint32_t* __restrict__ sorted_pos)
{
    for (uint32_t p = blockIdx.x * blockDim.x + threadIdx.x; p < n; p += gridDim.x * blockDim.x) {
        const uint32_t r = __ldg(&order[p]);
        distinct[p] = __ldg(&key[r]);
        counts[p] = (uint32_t)__ldg(&cnt[r]);
        sorted_pos[p] = r;
    }
}

// ---------------------------------------------------------------------------------------------------
// lookup_assign32_kernel: the per-read gather for rows outside any read map (bdg_assign_lookup32).  Every valid row's barcode is
// searched in the ascending node array (MEM_PIV pivots in shared memory, then the window between two pivots, as member_kernel);
// its node's centre index gives the centre node and that node's barcode.  A valid row whose barcode is no node counts as missing.
// 4 + 1 B in and 5 B out per row, plus the search (L2-resident for the node arrays of a correction step).
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(NT) lookup_assign32_kernel(const uint32_t* __restrict__ sorted, uint32_t N, const int32_t* __restrict__ centre_idx,
                                                             const uint32_t* __restrict__ ranks, const uint8_t* __restrict__ valid, uint64_t R,
                                                             uint32_t* __restrict__ out, uint8_t* __restrict__ out_has,
                                                             unsigned long long* __restrict__ counters /* [0] assigned, [1] missing */)
{
    __shared__ uint32_t s_p[MEM_PIV];
    const uint64_t step = ((uint64_t)N + MEM_PIV - 1) / MEM_PIV;
    for (int p = threadIdx.x; p < MEM_PIV; p += NT) {
        const uint64_t i = (uint64_t)p * step;
        s_p[p] = __ldg(&sorted[i < N ? i : N - 1]);
    }
    __syncthreads();
    unsigned long long assigned = 0, missing = 0;
    for (uint64_t i = (uint64_t)blockIdx.x * NT + threadIdx.x; i < R; i += (uint64_t)gridDim.x * NT) {
        uint32_t v = 0;
        uint8_t h = 0;
        if (!valid || __ldg(&valid[i])) {
            const uint32_t q = __ldg(&ranks[i]);
            int lo = 0, hi = MEM_PIV;
#pragma unroll
            for (int it = 0; it < 10; it++) {
                const int mid = (lo + hi) >> 1;
                if (s_p[mid] <= q) lo = mid; else hi = mid;
            }
            uint64_t l = (uint64_t)lo * step, u = min((uint64_t)N, l + step);
            if (l >= N) { l = N - 1; u = N; }
            while (l < u) {
                const uint64_t mid = (l + u) >> 1;
                if (__ldg(&sorted[mid]) < q) l = mid + 1; else u = mid;
            }
            if (l < N && __ldg(&sorted[l]) == q) {
                const int32_t c = __ldg(&centre_idx[l]);
                if (c >= 0 && (uint32_t)c < N) { v = __ldg(&sorted[c]); h = 1; }
            } else {
                missing++;
            }
        }
        out[i] = v;
        out_has[i] = h;
        assigned += h;
    }
    for (int o = 16; o; o >>= 1) {
        assigned += __shfl_down_sync(0xffffffffu, assigned, o);
        missing += __shfl_down_sync(0xffffffffu, missing, o);
    }
    if ((threadIdx.x & 31) == 0) {
        if (assigned) atomicAdd(&counters[0], assigned);
        if (missing) atomicAdd(&counters[1], missing);
    }
}

// ---------------------------------------------------------------------------------------------------
// Rows f-1 / f-2 with the per-read arrays staying on the device: bdg_dedup_reads compacts the valid rows (valid bytes +
// their exclusive scan), dedups them as above and keeps read -> first-seen position resident; bdg_assign_reads32 then
// turns the clustering result into the centre of every input row (barcode_graph.py:322-329 + 395-404) with two
// gathers.  HBM bound: 4 + 1 + 4 B in and 5 B out per row plus one random 5-byte read of the per-barcode table.
// ---------------------------------------------------------------------------------------------------
struct NonZero {
    __host__ __device__ __forceinline__ uint32_t operator()(const uint8_t& v) const { return v ? 1u : 0u; }
};

__global__ void compact_valid_kernel(const uint32_t* __restrict__ ranks, const uint8_t* __restrict__ valid, const uint32_t* __restrict__ excl,
                                     uint32_t n, uint32_t* __restrict__ out)
{
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
        if (__ldg(&valid[i])) out[__ldg(&excl[i])] = __ldg(&ranks[i]);
}

// centre value + "has a centre" byte of every distinct barcode in first-seen order: node = order[p]; centre_idx[node] >= 0 ->
// barcode of that node
__global__ void centre_of_distinct32_kernel(const int32_t* __restrict__ centre_idx, const uint32_t* __restrict__ order,
                                            const uint32_t* __restrict__ node_key, uint32_t n, uint32_t* __restrict__ out, uint8_t* __restrict__ has)
{
    for (uint32_t p = blockIdx.x * blockDim.x + threadIdx.x; p < n; p += gridDim.x * blockDim.x) {
        const int32_t c = __ldg(&centre_idx[__ldg(&order[p])]);
        const bool ok = c >= 0 && (uint32_t)c < n;
        out[p] = ok ? __ldg(&node_key[c]) : 0u;
        has[p] = ok ? 1 : 0;
    }
}

__global__ void assign_reads32_kernel(const uint32_t* __restrict__ centre_of_distinct, const uint8_t* __restrict__ has_of_distinct,
                                      const uint32_t* __restrict__ read_to_distinct, const uint8_t* __restrict__ valid,
                                      const uint32_t* __restrict__ excl, uint32_t n_rows, uint32_t* __restrict__ out, uint8_t* __restrict__ out_has,
                                      unsigned long long* __restrict__ n_assigned)
{
    unsigned long long mine = 0;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n_rows; i += gridDim.x * blockDim.x) {
        uint32_t v = 0;
        uint8_t h = 0;
        if (!valid || __ldg(&valid[i])) {
            const uint32_t p = __ldg(&read_to_distinct[valid ? __ldg(&excl[i]) : i]);
            v = __ldg(&centre_of_distinct[p]);
            h = __ldg(&has_of_distinct[p]);
        }
        out[i] = v;
        out_has[i] = h;
        mine += h;
    }
    for (int o = 16; o; o >>= 1) mine += __shfl_down_sync(0xffffffffu, mine, o);
    if ((threadIdx.x & 31) == 0 && mine) atomicAdd(n_assigned, mine);
}

// ---- centre selection on the device (reference barcode_graph.py:252-258): sum of the first counts, the barcodes above the
//      cutoff (cub select keeps their first-seen order), their count-descending stable order (cub radix sort of ~count) ----
__global__ void sum_first_kernel(const uint32_t* __restrict__ counts, uint32_t n, unsigned long long* __restrict__ out)
{
    unsigned long long mine = 0;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) mine += __ldg(&counts[i]);
    for (int o = 16; o; o >>= 1) mine += __shfl_down_sync(0xffffffffu, mine, o);
    if ((threadIdx.x & 31) == 0 && mine) atomicAdd(out, mine);
}

struct CountAbove {
    const uint32_t* counts;
    uint32_t thr;
    __host__ __device__ __forceinline__ bool operator()(const uint32_t& p) const { return counts[p] > thr; }
};

struct CountIs {
    const uint32_t* counts;
    uint32_t v;
    __host__ __device__ __forceinline__ bool operator()(const uint32_t& p) const { return counts[p] == v; }
};

__global__ void centres_keys_kernel(const uint32_t* __restrict__ pos, const uint32_t* __restrict__ counts, uint32_t n, uint32_t* __restrict__ keys)
{
    for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; j < n; j += gridDim.x * blockDim.x) keys[j] = ~__ldg(&counts[__ldg(&pos[j])]);
}

__global__ void centres_gather_kernel(const uint32_t* __restrict__ pos, const uint32_t* __restrict__ distinct, const uint32_t* __restrict__ counts,
                                      uint32_t n, uint32_t* __restrict__ top_ranks, uint32_t* __restrict__ top_counts)
{
    for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; j < n; j += gridDim.x * blockDim.x) {
        const uint32_t p = __ldg(&pos[j]);
        top_ranks[j] = __ldg(&distinct[p]);
        top_counts[j] = __ldg(&counts[p]);
    }
}

// nodes that have an edge but are no centre (what `len(graph.edges.keys())`, badger.py:131, counts beside the centres)
__global__ void count_has_edge_kernel(const uint8_t* __restrict__ level, uint32_t n, unsigned long long* __restrict__ out)
{
    unsigned long long mine = 0;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const uint8_t l = __ldg(&level[i]);
        mine += (l != 255 && l != 0) ? 1 : 0;                 // 254 = untouched with an edge; 1, 2 = joined over an edge
    }
    for (int o = 16; o; o >>= 1) mine += __shfl_down_sync(0xffffffffu, mine, o);
    if ((threadIdx.x & 31) == 0 && mine) atomicAdd(out, mine);
}

// ---------------------------------------------------------------------------------------------------
// Clustering rounds (row f-3, reference barcode_graph.py:279-301): level-synchronous and edge-parallel.
//   round i: every edge (u,v), both directions: if u joined a centre at level i-1 and v is still free, u's
//   centre claims v (atomicMin / atomicMax of the centre index);  then every claimed v joins the centre if all
//   claims of this round agree, and is evicted (centre -1) if two different centres claimed it - exactly the
//   reference's same-round conflict rule, which does not depend on the adjacency order (SURVEY.md 4).
// Nodes are positions in the sorted distinct-barcode array; centre_idx: -2 free, -1 evicted, else a node.
// HBM/L2-latency bound: per edge and round two index pairs in, a few random 4-byte reads.
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t lower_bound_u32(const uint32_t* __restrict__ v, uint32_t n, uint32_t x)
{
    uint32_t lo = 0, hi = n;
    while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        if (__ldg(&v[mid]) < x) lo = mid + 1; else hi = mid;
    }
    return lo;
}

__global__ void cluster_init_kernel(int32_t* __restrict__ centre_idx, uint8_t* __restrict__ level, int32_t* __restrict__ cmin,
                                    int32_t* __restrict__ cmax, uint32_t n)
{
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        centre_idx[i] = -2; level[i] = 255; cmin[i] = 0x7FFFFFFF; cmax[i] = -1;
    }
}

__global__ void cluster_seed_kernel(const uint32_t* __restrict__ sorted, uint32_t n, const uint32_t* __restrict__ centres, uint32_t n_centres,
                                    int32_t* __restrict__ centre_idx, uint8_t* __restrict__ level)
{
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n_centres; i += gridDim.x * blockDim.x) {
        const uint32_t c = __ldg(&centres[i]);
        const uint32_t p = lower_bound_u32(sorted, n, c);
        if (p < n && __ldg(&sorted[p]) == c) { centre_idx[p] = (int32_t)p; level[p] = 0; }   // centres that were never observed have no node
    }
}

// top[h] = first node whose barcode has the high half h (h = 0 .. 65536): the node of a barcode is then found in a run of
// N / 65536 entries instead of all N (10 probes instead of 26 at N = 5e7)
__global__ void top_start_kernel(const uint32_t* __restrict__ sorted, uint32_t n, uint32_t* __restrict__ top)
{
    for (uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; j <= n; j += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t k_hi = j < n ? (__ldg(&sorted[j]) >> 16) : 65536u;
        const uint32_t k_lo = j > 0 ? (__ldg(&sorted[j - 1]) >> 16) + 1u : 0u;
        for (uint32_t k = k_lo; k <= k_hi; k++) top[k] = (uint32_t)j;
    }
}

constexpr uint8_t LEVEL_NONE = 255, LEVEL_HAS_EDGE = 254;
// An end point that is not a node (a value absent from `sorted`) becomes NO_NODE at both ends of its edge; cluster_mark_kernel
// raises the error flag for it and the claim kernel skips it.
constexpr uint32_t NO_NODE = 0xFFFFFFFFu;

__device__ __forceinline__ uint32_t node_of(const uint32_t* __restrict__ sorted, const uint32_t* __restrict__ top, uint32_t v)
{
    uint32_t lo = __ldg(&top[v >> 16]), hi = __ldg(&top[(v >> 16) + 1u]);
    const uint32_t end = hi;
    while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        if (__ldg(&sorted[mid]) < v) lo = mid + 1; else hi = mid;
    }
    return (lo < end && __ldg(&sorted[lo]) == v) ? lo : NO_NODE;
}

// barcode values of an edge list -> node indices (in place when out == in).  Runs on the device that holds the edges.
__global__ void cluster_index_kernel(const uint32_t* __restrict__ sorted, const uint32_t* __restrict__ top, const uint32_t* ea, const uint32_t* eb,
                                     uint64_t n_edges, uint32_t* oa, uint32_t* ob)
{
    for (uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n_edges; e += (uint64_t)gridDim.x * blockDim.x) {
        uint32_t ia = node_of(sorted, top, ea[e]), ib = node_of(sorted, top, eb[e]);
        if (ia == NO_NODE || ib == NO_NODE) ia = ib = NO_NODE;
        oa[e] = ia;
        ob[e] = ib;
    }
}

// mark both ends of every edge "has an edge" (level 254; centres keep their 0, later rounds overwrite the mark of whoever they reach)
__global__ void cluster_mark_kernel(const uint32_t* __restrict__ ia, const uint32_t* __restrict__ ib, uint64_t n_edges, uint8_t* __restrict__ level,
                                    unsigned int* __restrict__ bad)
{
    for (uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n_edges; e += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t u = __ldg(&ia[e]), v = __ldg(&ib[e]);
        if (u == NO_NODE) { *bad = 1u; continue; }
        if (level[u] == LEVEL_NONE) level[u] = LEVEL_HAS_EDGE;                 // every writer stores the same value
        if (level[v] == LEVEL_NONE) level[v] = LEVEL_HAS_EDGE;
    }
}

__global__ void cluster_claim_kernel(const uint32_t* __restrict__ ia, const uint32_t* __restrict__ ib, uint64_t n_edges, int round,
                                     const int32_t* __restrict__ centre_idx, const uint8_t* __restrict__ level,
                                     int32_t* __restrict__ cmin, int32_t* __restrict__ cmax)
{
    for (uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n_edges; e += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t u = __ldg(&ia[e]), v = __ldg(&ib[e]);
        if (u == NO_NODE) continue;
        const int32_t cu = centre_idx[u], cv = centre_idx[v];
        if (cu >= 0 && cv == -2 && level[u] == round - 1) { atomicMin(&cmin[v], cu); atomicMax(&cmax[v], cu); }
        if (cv >= 0 && cu == -2 && level[v] == round - 1) { atomicMin(&cmin[u], cv); atomicMax(&cmax[u], cv); }
    }
}

__global__ void cluster_resolve_kernel(int32_t* __restrict__ centre_idx, uint8_t* __restrict__ level, int32_t* __restrict__ cmin,
                                       int32_t* __restrict__ cmax, uint32_t n, int round)
{
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const int32_t lo = cmin[i];
        if (lo != 0x7FFFFFFF) {
            const bool single = lo == cmax[i];
            centre_idx[i] = single ? lo : -1;
            level[i] = single ? (uint8_t)round : LEVEL_HAS_EDGE;             // evicted: still a node with edges
            cmin[i] = 0x7FFFFFFF; cmax[i] = -1;
        }
    }
}

}  // namespace bdg
