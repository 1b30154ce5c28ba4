// Host build of badger_b200/csrc/bdg_seed3.cuh for the CPU-side unit tests (tests/test_seed3_host.py).
// Test infrastructure: lets the t = 3 seed scheme, its hand-over and the join passes be checked against the oracle without a GPU.
#include "../badger_b200/csrc/bdg_seed3.cuh"
#include <stddef.h>
#include <algorithm>
#include <vector>

static bdg::Seed3Scheme g_s3;

extern "C" {
int shim3_scheme(const int* bases, int nblocks)          // returns the number of conditions, -1 if the layout is refused
{
    if (!bdg::seed3_scheme_build(g_s3, bases, nblocks)) return -1;
    return g_s3.nconds;
}
int shim3_nself(void) { return g_s3.nself; }
int shim3_nsets(void) { return g_s3.nsets; }
int shim3_key_bits(int c) { return g_s3.ka[c].key_bits; }
int shim3_set(int c) { return g_s3.cond[c].set; }
int shim3_self(int c) { return g_s3.cond[c].self; }
// first (condition, orientation) by the definition and by the kernel's walk over the flags
void shim3_first(const uint32_t* a, const uint32_t* b, size_t n, int32_t* slow, int32_t* fast)
{
    for (size_t i = 0; i < n; i++) {
        slow[i] = bdg::seed3_first_slow(g_s3, a[i], b[i]);
        fast[i] = bdg::seed3_first(g_s3, a[i], b[i]);
    }
}
// number of (condition, orientation) pairs the pair meets
void shim3_hits(const uint32_t* a, const uint32_t* b, size_t n, int32_t* hits)
{
    for (size_t i = 0; i < n; i++) {
        int h = 0;
        for (int c = 0; c < g_s3.nconds; c++) h += bdg::seed3_pred(g_s3, c, a[i], b[i]) + (!g_s3.cond[c].self && bdg::seed3_pred(g_s3, c, b[i], a[i]));
        hits[i] = h;
    }
}
// Every 16-mer within three edit operations of a (an insertion keeps the first 16 bases, a deletion appends each of the four
// bases): out[0] distinct words, [1] of them with D <= 3, [2] D <= 3 words that meet no condition in either orientation,
// [3] D <= 3 words whose quick test fails, [4] words where seed3_first and the definition disagree (the definition is evaluated
// on every check_stride-th D <= 3 word and on every word seed3_first finds unmet).
static void neigh_step(const std::vector<uint32_t>& in, std::vector<uint32_t>& out)
{
    for (uint32_t w : in) {
        for (int i = 0; i < 16; i++)
            for (uint32_t c = 1; c < 4; c++) out.push_back(w ^ (c << (2 * i)));
        for (int i = 0; i <= 16; i++)                       // insert base c in front of column i, keep 16 bases
            for (uint32_t c = 0; c < 4; c++) {
                const uint32_t lo = i ? (w & bdg::low_mask(2 * i)) : 0u;
                out.push_back(i == 16 ? w : (lo | (c << (2 * i)) | ((w >> (2 * i)) << (2 * i + 2))));
            }
        for (int i = 0; i < 16; i++)                        // delete column i, append base c
            for (uint32_t c = 0; c < 4; c++) {
                const uint32_t lo = i ? (w & bdg::low_mask(2 * i)) : 0u;
                const uint32_t hi = i < 15 ? ((w >> (2 * i + 2)) << (2 * i)) : 0u;
                out.push_back(lo | (hi & bdg::low_mask(30)) | (c << 30));
            }
    }
    std::sort(out.begin(), out.end());
    out.erase(std::unique(out.begin(), out.end()), out.end());
}
void shim3_neighbourhood(uint32_t a, int check_stride, unsigned long long* out)
{
    std::vector<uint32_t> cur{a}, next, all{a};
    for (int step = 0; step < 3; step++) {
        next.clear();
        neigh_step(cur, next);
        all.insert(all.end(), next.begin(), next.end());
        cur.swap(next);
    }
    std::sort(all.begin(), all.end());
    all.erase(std::unique(all.begin(), all.end()), all.end());
    for (int k = 0; k < 5; k++) out[k] = 0;
    out[0] = all.size();
    unsigned long long near = 0;
    for (uint32_t b : all) {
        if (b == a) continue;
        const uint32_t x = a < b ? a : b, y = a < b ? b : a;
        if (bdg::dist3_min(x, y) > 3) continue;
        out[1]++;
        if (!bdg::quick3_pass(x, y)) out[3]++;
        const int fast = bdg::seed3_first(g_s3, x, y);
        if (fast == bdg::SEED3_NONE || (near++ % (unsigned long long)check_stride) == 0) {
            const int slow = bdg::seed3_first_slow(g_s3, x, y);
            if (slow == bdg::SEED3_NONE) out[2]++;
            if (slow != fast) out[4]++;
        }
    }
}
void shim3_quick(const uint32_t* a, const uint32_t* b, size_t n, uint8_t* out)
{
    for (size_t i = 0; i < n; i++) out[i] = bdg::quick3_pass(a[i], b[i]);
}
// The t = 3 join passes emulated: per condition both sides are sorted by their join key, equal-key buckets are paired, and a
// candidate goes through the very checks of the kernel (quick test, dist3_min, seed3_first, qgram_score).  Returns the number of
// edges (first `cap` stored).  stats: 0 pairs of the buckets, 1 pairs that pass the quick test, 2 of those with D <= 3,
// 3 of those handed to this pass, 4 edges.
size_t shim3_join_emulate(const uint32_t* s, size_t n, uint32_t* oa, uint32_t* ob, uint8_t* od, size_t cap, unsigned long long* stats)
{
    const bdg::Seed3Scheme& S = g_s3;
    size_t cnt = 0;
    for (int k = 0; k < 5; k++) stats[k] = 0;
    std::vector<uint32_t> rows(s, s + n), cols(s, s + n);
    for (int c = 0; c < S.nconds; c++) {
        const bdg::SeedKey A = S.ka[c], B = S.kb[c];
        std::stable_sort(rows.begin(), rows.end(), [&](uint32_t p, uint32_t q) { return bdg::seed_key(p, A) < bdg::seed_key(q, A); });
        std::stable_sort(cols.begin(), cols.end(), [&](uint32_t p, uint32_t q) { return bdg::seed_key(p, B) < bdg::seed_key(q, B); });
        size_t lo = 0, hi = 0;
        for (size_t r = 0; r < n; r++) {
            const uint32_t x = rows[r], ka = bdg::seed_key(x, A);
            while (lo < n && bdg::seed_key(cols[lo], B) < ka) lo++;
            if (hi < lo) hi = lo;
            while (hi < n && bdg::seed_key(cols[hi], B) <= ka) hi++;
            for (size_t j = lo; j < hi; j++) {
                const uint32_t y = cols[j];
                if (S.cond[c].self && !(x < y)) continue;          // a symmetric condition pairs each couple once
                stats[0]++;
                if (x == y || !bdg::quick3_pass(x, y)) continue;
                stats[1]++;
                const uint32_t a = x < y ? x : y, b = x < y ? y : x;
                const int d = bdg::dist3_min(a, b);
                if (d > 3) continue;
                stats[2]++;
                if (bdg::seed3_first(S, a, b) != 2 * c + (x < y || S.cond[c].self ? 0 : 1)) continue;
                stats[3]++;
                if (bdg::qgram_score(a, b) < bdg::qgram_threshold(3)) continue;
                stats[4]++;
                if (cnt < cap) { oa[cnt] = a; ob[cnt] = b; od[cnt] = (uint8_t)d; }
                cnt++;
            }
        }
    }
    return cnt;
}
}
