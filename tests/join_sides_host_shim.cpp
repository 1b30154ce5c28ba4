// Host build of the t = 2 join's one-sided filter and side-aware hand-over (bdg_seed.cuh) for tests/test_join_sides_host.py.
// Test infrastructure: the kernel's per-pair functions (join2_quick, seed_side_bits, seed_flags) and the table the driver
// uploads (seed_lut_build_sides), checked against their definitions and against the oracle's edge set without a GPU.
#include "../badger_b200/csrc/bdg_seed.cuh"
#include <stddef.h>
#include <algorithm>
#include <vector>

static bdg::SeedScheme g_scheme;
static std::vector<uint8_t> g_lut, g_lut_sides;

extern "C" {
int shim_scheme(const int* bases, int nblocks)          // returns the number of conditions, -1 if the layout is refused
{
    if (!bdg::seed_scheme_build(g_scheme, bases, nblocks)) return -1;
    g_lut.assign((size_t)1 << g_scheme.nflags, 0);
    bdg::seed_lut_build(g_scheme, g_lut.data());
    g_lut_sides.assign((size_t)1 << (g_scheme.nflags + 2), 0);
    bdg::seed_lut_build_sides(g_scheme, g_lut_sides.data());
    return g_scheme.nconds;
}
int shim_nflags(void) { return g_scheme.nflags; }
// condition c: number of blocks, their indices and diagonals; returns whether it is symmetric
int shim_cond(int c, int* nf, int* blk, int* d)
{
    *nf = g_scheme.cond[c].nf;
    for (int k = 0; k < *nf; k++) { blk[k] = g_scheme.cond[c].blk[k]; d[k] = g_scheme.cond[c].d[k]; }
    return g_scheme.cond[c].self;
}
void shim_tables(uint8_t* lut, uint8_t* lut_sides)
{
    std::copy(g_lut.begin(), g_lut.end(), lut);
    std::copy(g_lut_sides.begin(), g_lut_sides.end(), lut_sides);
}
// per pair (a < b): owner by the definition, owner through the table at the index join_process reads, the side bits, and
// whether the owner's own pass lets the pair through its quick test (bit 0) and meets the owner's key (bit 1)
void shim_owner(const uint32_t* a, const uint32_t* b, size_t n, uint8_t* slow, uint8_t* fast, uint8_t* sides, uint8_t* passes)
{
    const bdg::SeedScheme& S = g_scheme;
    for (size_t i = 0; i < n; i++) {
        const uint32_t p = a[i], q = b[i];
        slow[i] = (uint8_t)bdg::seed_first_sides_slow(S, p, q);
        sides[i] = (uint8_t)bdg::seed_side_bits(p, q);
        fast[i] = g_lut_sides[bdg::seed_flags(S, p, q) | (uint32_t)sides[i] << S.nflags];
        passes[i] = 0;
        if (slow[i] == bdg::SEED_NONE) continue;
        const int c = slow[i] >> 1, o = slow[i] & 1;
        const uint32_t x = o ? q : p, y = o ? p : q;             // the owner's row and column
        bool pass;
        if (S.cond[c].self)       // the bucket holds the pair in either order
            pass = bdg::join2_quick<false>(x, y, y >> 2, y << 2, 1u, 0xFFFFFFFFu) && bdg::join2_quick<false>(y, x, x >> 2, x << 2, 1u, 0xFFFFFFFFu);
        else
            pass = bdg::join2_quick<true>(x, y, y >> 2, y << 2, 1u, 0xFFFFFFFFu);
        passes[i] = (uint8_t)((pass ? 1 : 0) | (bdg::seed_pred(S, c, x, y) ? 2 : 0));
    }
}
// the kernel's filter of one orientation: out[i] = join2_quick<shf>(x, y) | the old three-diagonal quick test << 1
void shim_filter(int shf, const uint32_t* x, const uint32_t* y, size_t n, uint8_t* out)
{
    for (size_t i = 0; i < n; i++) {
        const bool f = shf ? bdg::join2_quick<true>(x[i], y[i], y[i] >> 2, y[i] << 2, 1u, 0xFFFFFFFFu)
                           : bdg::join2_quick<false>(x[i], y[i], y[i] >> 2, y[i] << 2, 1u, 0xFFFFFFFFu);
        out[i] = (uint8_t)((f ? 1 : 0) | (bdg::quick_pass(x[i], y[i], 2) ? 2 : 0));
    }
}
// The join passes emulated with the kernel's per-pair functions: per condition both sides are bucketed by their join key in a
// stable order (so the input order decides the order inside a bucket, as the atomics do on the device), a symmetric condition
// pairs each couple of a bucket once in bucket order, and a pair goes through join2_quick<shifted>, dist_small, the side-aware
// hand-over table and the score.  Returns the number of edges (first `cap` stored).  stats: [0] pairs of the buckets,
// [1] candidates, [2] of those with D <= 2, [3] of those handed to this pass, [4] edges, [5] candidates of the three-diagonal
// quick test on the same pairs.
size_t shim_join_emulate(const uint32_t* s, size_t n, uint32_t* oa, uint32_t* ob, uint8_t* od, size_t cap, unsigned long long* stats)
{
    const bdg::SeedScheme& S = g_scheme;
    size_t cnt = 0;
    for (int k = 0; k < 6; k++) stats[k] = 0;
    std::vector<uint32_t> rows, cols;
    for (int c = 0; c < S.nconds; c++) {
        const bdg::SeedKey A = S.ka[c], B = S.kb[c];
        const bool self = S.cond[c].self != 0;
        rows.assign(s, s + n);
        cols.assign(s, s + n);
        std::stable_sort(rows.begin(), rows.end(), [&](uint32_t p, uint32_t q) { return bdg::seed_key(p, A) < bdg::seed_key(q, A); });
        std::stable_sort(cols.begin(), cols.end(), [&](uint32_t p, uint32_t q) { return bdg::seed_key(p, B) < bdg::seed_key(q, B); });
        size_t lo = 0, hi = 0;
        for (size_t r = 0; r < n; r++) {
            const uint32_t x = rows[r], ka = bdg::seed_key(x, A);
            while (lo < n && bdg::seed_key(cols[lo], B) < ka) lo++;
            if (hi < lo) hi = lo;
            while (hi < n && bdg::seed_key(cols[hi], B) <= ka) hi++;
            for (size_t j = self ? std::max(lo, r + 1) : lo; j < hi; j++) {
                const uint32_t y = cols[j];
                if (x == y) continue;
                stats[0]++;
                stats[5] += bdg::quick_pass(x, y, 2);
                const bool pass = self ? bdg::join2_quick<false>(x, y, y >> 2, y << 2, 1u, 0xFFFFFFFFu)
                                       : bdg::join2_quick<true>(x, y, y >> 2, y << 2, 1u, 0xFFFFFFFFu);
                if (!pass) continue;
                stats[1]++;
                const uint32_t a = std::min(x, y), b = std::max(x, y);
                const int d = bdg::dist_small(a, b, false, true);
                if (d > 2) continue;
                stats[2]++;
                const uint32_t idx = bdg::seed_flags(S, a, b) | bdg::seed_side_bits(a, b) << S.nflags;
                if (g_lut_sides[idx] != 2 * c + (self || x < y ? 0 : 1)) continue;
                stats[3]++;
                if (bdg::qgram_score(a, b) < bdg::qgram_threshold(2)) continue;
                stats[4]++;
                if (cnt < cap) { oa[cnt] = a; ob[cnt] = b; od[cnt] = (uint8_t)d; }
                cnt++;
            }
        }
    }
    return cnt;
}
}
