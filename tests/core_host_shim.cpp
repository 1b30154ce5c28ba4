// Host build of badger_b200/csrc/bdg_core.cuh for the CPU-side unit tests (tests/test_core_host.py).
// Test infrastructure: lets the per-pair device arithmetic be checked against the oracle without a GPU.
#include "../badger_b200/csrc/bdg_seed.cuh"
#include <stddef.h>
#include <algorithm>
#include <vector>

extern "C" {
void shim_pairs(const uint32_t* a, const uint32_t* b, size_t n, uint8_t* pre1, uint8_t* pre2, uint8_t* dsmall,
                uint8_t* dplain, uint8_t* dfull, uint8_t* da15, uint8_t* db15, uint8_t* S, uint64_t* mult)
{
    for (size_t i = 0; i < n; i++) {
        pre1[i] = bdg::prefilter_t1(a[i], b[i]);
        pre2[i] = bdg::prefilter_t2(a[i], b[i]);
        dsmall[i] = (uint8_t)bdg::dist_small(a[i], b[i], false);
        if (bdg::dist_small(a[i], b[i], false, true) != (int)dsmall[i]) dsmall[i] = 200;    // without its quick reject: the same value
        dplain[i] = (uint8_t)bdg::dist_small(a[i], b[i], true);
        bdg::Dist3 r = bdg::myers3(a[i], b[i]);
        dfull[i] = (uint8_t)r.full; da15[i] = (uint8_t)r.a15; db15[i] = (uint8_t)r.b15;
        S[i] = (uint8_t)bdg::qgram_score(a[i], b[i], &mult[i]);
    }
}
int shim_edge(uint32_t a, uint32_t b, int t) { return bdg::edge_dist(a, b, t); }
// split prefilters of the tiled edge kernel: light (per pair) and top (excluded per tile)
void shim_split(const uint32_t* a, const uint32_t* b, size_t n, uint8_t* l1, uint8_t* t1, uint8_t* l2, uint8_t* t2)
{
    for (size_t i = 0; i < n; i++) {
        l1[i] = bdg::t1_light(a[i], b[i]); t1[i] = bdg::t1_top(a[i], b[i]);
        l2[i] = bdg::t2_light(a[i], b[i]); t2[i] = bdg::t2_top(a[i], b[i]);
    }
}
void shim_pass_pred(int t, const uint32_t* a, const uint32_t* b, size_t n, uint8_t* mask /* bit p = pass p fires */)
{
    for (size_t i = 0; i < n; i++) {
        uint8_t m = 0;
        for (int p = 0; p < bdg::n_passes(t); p++) {
            const bool f = bdg::pass_pred(t, p, a[i], b[i]);
            const int r = bdg::pass_rot(t, p);
            if (f != bdg::pass_pred_rot(t, p, bdg::rotl32(a[i], r), bdg::rotl32(b[i], r))) m |= 0x80;   // must agree
            if (f) m |= (uint8_t)(1u << p);
        }
        mask[i] = m;
    }
}
int shim_pass_possible(int t, int p, uint32_t alo, uint32_t ahi, uint32_t blo, uint32_t bhi)
{
    return bdg::pass_possible(t, p, alo, ahi, blo, bhi);
}
void shim_quick(int t, const uint32_t* a, const uint32_t* b, size_t n, uint8_t* out)
{
    for (size_t i = 0; i < n; i++) out[i] = bdg::quick_pass(a[i], b[i], t);
}
void shim_quick_any(int t, const uint32_t* a, const uint32_t* b, size_t n, uint8_t* out)
{
    for (size_t i = 0; i < n; i++) out[i] = bdg::quick_pass_any(a[i], b[i], t);
}
int shim_top_possible(int t, uint32_t alo, uint32_t ahi, uint32_t blo, uint32_t bhi)
{
    return t == 1 ? bdg::t1_top_possible(alo, ahi, blo, bhi) : bdg::t2_top_possible(alo, ahi, blo, bhi);
}

// ---- multi-block seeds (bdg_seed.cuh): scheme tables, hand-over table, sort forms, and the join passes emulated on the host
static bdg::SeedScheme g_scheme;
static std::vector<uint8_t> g_lut;
int shim_scheme(const int* bases, int nblocks)          // returns the number of conditions, -1 if the layout is refused
{
    if (!bdg::seed_scheme_build(g_scheme, bases, nblocks)) return -1;
    g_lut.assign((size_t)1 << g_scheme.nflags, 0);
    bdg::seed_lut_build(g_scheme, g_lut.data());
    return g_scheme.nconds;
}
int shim_scheme_nself(void) { return g_scheme.nself; }
int shim_scheme_key_bits(int c) { return g_scheme.ka[c].key_bits; }
int shim_scheme_row_sort(int c) { return g_scheme.cond[c].row_sort; }
int shim_scheme_nsets(void) { return g_scheme.nsets; }
int shim_scheme_set_first(int k) { return g_scheme.set_first[k]; }
// first (condition, orientation) by the definition and by the table over the block-match flags
void shim_scheme_first(const uint32_t* a, const uint32_t* b, size_t n, uint8_t* slow, uint8_t* fast)
{
    for (size_t i = 0; i < n; i++) {
        slow[i] = (uint8_t)bdg::seed_first_slow(g_scheme, a[i], b[i]);
        fast[i] = g_lut[bdg::seed_flags(g_scheme, a[i], b[i])];
        if (bdg::seed_flags(g_scheme, a[i], b[i]) != bdg::seed_flags_slow(g_scheme, a[i], b[i])) fast[i] = 254;   // must agree
    }
}
void shim_qgram_compact(const uint32_t* a, const uint32_t* b, size_t n, uint8_t* full, uint8_t* compact)
{
    for (size_t i = 0; i < n; i++) { full[i] = (uint8_t)bdg::qgram_score(a[i], b[i]); compact[i] = (uint8_t)bdg::qgram_score_compact(a[i], b[i]);
                                     if (bdg::qgram_score_near(a[i], b[i]) + bdg::qgram_score_far(a[i], b[i]) != (int)full[i]) compact[i] = 255; }
}
// The posting-list form of a-5 (kmer_post_kernel) on the host: buckets of string ids per 6-mer, a query walks the buckets of its
// distinct 6-mers and a hit is emitted from the bucket of the first query position whose 6-mer occurs in the entry.
size_t shim_kmer_post_emulate(const uint32_t* q, size_t Q, const uint32_t* wl, size_t W, int min_kmers, uint32_t* hq, uint32_t* hw, uint8_t* cnt,
                              size_t cap, unsigned long long* evaluated)
{
    std::vector<std::vector<uint32_t>> bucket(4096);
    for (size_t i = 0; i < W; i++)
        for (int p = 0; p <= 10; p++)
            if (!bdg::kmer_seen_before(wl[i], p)) bucket[(wl[i] >> (2 * p)) & 0xFFFu].push_back((uint32_t)i);
    size_t n = 0;
    *evaluated = 0;
    for (size_t x = 0; x < Q; x++)
        for (int p = 0; p <= 10; p++) {
            if (bdg::kmer_seen_before(q[x], p)) continue;
            for (uint32_t wi : bucket[(q[x] >> (2 * p)) & 0xFFFu]) {
                uint32_t marks = 0;
                const int s = bdg::qgram_score_marks(q[x], wl[wi], &marks);
                (*evaluated)++;
                if (s != bdg::qgram_score(q[x], wl[wi])) return (size_t)-1;
                if (s >= min_kmers && (marks & ((1u << (2 * p)) - 1u)) == 0) {
                    if (n < cap) { hq[n] = (uint32_t)x; hw[n] = wi; cnt[n] = (uint8_t)s; }
                    n++;
                }
            }
        }
    return n;
}
void shim_scheme_keys(int c, const uint32_t* a, const uint32_t* b, size_t n, uint32_t* ka, uint32_t* kb, uint8_t* pred)
{
    for (size_t i = 0; i < n; i++) {
        ka[i] = bdg::seed_key(a[i], g_scheme.ka[c]); kb[i] = bdg::seed_key(b[i], g_scheme.kb[c]);
        pred[i] = bdg::seed_pred(g_scheme, c, a[i], b[i]);
    }
}
// The join passes emulated: per condition both sides are sorted by their join key, equal-key buckets are paired, and a candidate
// goes through the very checks of the kernel (quick test, dist_small, hand-over table, qgram_score).  Returns the number of
// edges (first `cap` stored).  stats[5 * (c + 1) + k], summed over the conditions in stats[k]: k = 0 pairs of the buckets
// (quick tests), 1 pairs that pass the quick test, 2 of those with D <= 2, 3 of those handed to this pass, 4 edges.
size_t shim_join_emulate(const uint32_t* s, size_t n, uint32_t* oa, uint32_t* ob, uint8_t* od, size_t cap, unsigned long long* stats)
{
    const bdg::SeedScheme& S = g_scheme;
    size_t cnt = 0;
    for (int k = 0; k < 5 * (S.nconds + 1); k++) stats[k] = 0;
    std::vector<uint32_t> rows(s, s + n), cols(s, s + n);
    for (int c = 0; c < S.nconds; c++) {
        unsigned long long* st = stats + 5 * (c + 1);
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
                st[0]++;
                if (x == y || !bdg::quick_pass(x, y, 2)) continue;
                st[1]++;
                const uint32_t a = x < y ? x : y, b = x < y ? y : x;
                const int d = bdg::dist_small(a, b, false, true);
                if (d > 2) continue;
                st[2]++;
                if (g_lut[bdg::seed_flags(S, a, b)] != 2 * c + (x < y ? 0 : 1)) continue;
                st[3]++;
                if (bdg::qgram_score(a, b) < bdg::qgram_threshold(2)) continue;
                st[4]++;
                if (cnt < cap) { oa[cnt] = a; ob[cnt] = b; od[cnt] = (uint8_t)d; }
                cnt++;
            }
        }
        for (int k = 0; k < 5; k++) stats[k] += st[k];
    }
    return cnt;
}
}
