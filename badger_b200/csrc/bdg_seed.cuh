// bdg_seed.cuh -- multi-block seeds for the t = 2 edge construction by sort-merge joins (bdg_join.cuh).
//
// What is searched (reference index.py:77-93 + barcode_graph.py:233-249): pairs a < b with D(a,b) <= 2 and S(a,b) >= 4.
// A NECESSARY condition for D <= 2, sharper than the single 5-base blocks of the sparse passes (bdg_core.cuh):
//   * cut a[0:15] into B blocks (column 15 is left out: the truncated variants of D drop it for free);
//   * an edit script of <= 2 operations touches <= 2 blocks (an insertion in front of a[i] is charged to the block holding
//     a[i]), so >= B-2 blocks are untouched and each of them equals a stretch of b on one diagonal;
//   * the lengths behind D differ by <= 1, so a script of <= 2 operations keeps its columns on the diagonals {0, +1} or on
//     {0, -1}, never on both sides, and the inverse script (b -> a) has the negated diagonals: under ONE of the two
//     labellings of the pair all diagonals are >= 0;
//   * block 0 has nothing in front of it (diagonal 0); two untouched blocks with no touched block between them share their
//     diagonal; across touched blocks the diagonal moves by at most one.
// A condition = a set of B-2 blocks with one diagonal (0 or +1) each, i.e. "these fields of x equal those fields of y": a
// plain key equality, found by sorting both sides by the key (the barcode rides along as the value) and pairing
// equal-key buckets.  Conditions whose diagonals
// are all 0 are symmetric ("self": one sort, each unordered couple once); the others pair (x, y) in both value orders.
//   B = 4 (4,4,4,3 bases): 13 conditions on 14/16 key bits;  B = 5 (3 bases each): 25 conditions on 18 key bits.
// A pair that meets several conditions is emitted by the FIRST (condition, orientation) in table order; that index is
// looked up in a table over the pair's block-match flags (seed_flags / seed_lut_build), built here on the host.  The join
// kernel tests a shifted condition's pairs on one diagonal side only (join2_quick), so its hand-over table also takes the
// pair's two side bits and names the first (condition, orientation) that meets the pair AND lets it through its filter
// (seed_side_bits, seed_first_sides_slow, seed_lut_build_sides).
//
// Everything is __host__ __device__: tests/test_core_host.py compiles this header with g++ and checks, against the oracle's
// distances, that the conditions are necessary for D <= 2, and that the emulated passes give the oracle's edge set;
// tests/test_join_sides_host.py does the same for the one-sided filter and the side-aware table.
#pragma once
#include "bdg_core.cuh"

namespace bdg {

constexpr int SEED_MAX_BLOCKS = 6;
constexpr int SEED_MAX_FIELDS = 4;
constexpr int SEED_MAX_CONDS = 48;
constexpr int SEED_MAX_FLAGS = 3 * SEED_MAX_BLOCKS;
constexpr uint8_t SEED_NONE = 255;

// How one side of a condition reads its join key off a barcode: field f = (v >> lo[f]) & mask[f], placed at bit at[f] of the key
// (field 0 lowest).  Unused fields have mask 0, so the extraction is four branch-free shift-and-mask steps.
struct SeedKey {
    uint8_t nf, key_bits;
    uint8_t lo[SEED_MAX_FIELDS], n[SEED_MAX_FIELDS], at[SEED_MAX_FIELDS];
    uint32_t mask[SEED_MAX_FIELDS];
};

BDG_HD uint32_t seed_key(uint32_t v, const SeedKey& k)
{
    uint32_t r = 0;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int f = 0; f < SEED_MAX_FIELDS; f++) r |= ((v >> k.lo[f]) & k.mask[f]) << k.at[f];
    return r;
}

struct SeedCond {
    uint8_t nf;                       // number of blocks in the condition
    uint8_t blk[SEED_MAX_FIELDS];     // ascending
    uint8_t d[SEED_MAX_FIELDS];       // diagonal of each block: 0 or 1 (x[block] == y[block columns + d])
    uint8_t self;                     // all diagonals 0
    uint8_t row_sort;                 // first condition with the same blocks (they follow one another and share the row order)
};

struct SeedScheme {
    int nblocks;
    uint8_t blo[SEED_MAX_BLOCKS], bn[SEED_MAX_BLOCKS];     // first bit / number of bits of every block
    int nconds, nself;                                     // nself of the conditions are symmetric (the first of every block set)
    SeedCond cond[SEED_MAX_CONDS];
    SeedKey ka[SEED_MAX_CONDS], kb[SEED_MAX_CONDS];        // join key of the row side (fields of x) / column side (fields of y)
    int nflags;                                            // bits of seed_flags: 3 per block
    uint32_t hi_mask, lo_mask;                             // top bit of every block / the other bits of the blocks
    uint32_t fmask[SEED_MAX_BLOCKS], fnet[SEED_MAX_BLOCKS]; // seed_flags: where block k's three flags sit in the zero-field word, and how far they move down
    int nsets;                                             // block sets, as in Seed3Scheme: the conditions of set s are
    uint16_t set_first[SEED_MAX_CONDS + 1];                // set_first[s] .. set_first[s + 1] - 1
};

// x[fields of condition c] == y[the same fields moved by their diagonals]
BDG_HD bool seed_pred(const SeedScheme& s, int c, uint32_t x, uint32_t y) { return seed_key(x, s.ka[c]) == seed_key(y, s.kb[c]); }

// first (condition, orientation) the pair meets, as 2 * c + o (o = 0: (x, y) = (a, b); o = 1: (x, y) = (b, a)), by the
// definition; SEED_NONE if none.  The kernels use the table form below.
BDG_HD int seed_first_slow(const SeedScheme& s, uint32_t a, uint32_t b)
{
    for (int c = 0; c < s.nconds; c++) {
        if (seed_pred(s, c, a, b)) return 2 * c;
        if (!s.cond[c].self && seed_pred(s, c, b, a)) return 2 * c + 1;
    }
    return SEED_NONE;
}

// Block-match flags of a pair, three bits per block k at bit 3k: a[block k] == b[block k] | a[block k] == b[block k moved one
// column up] << 1 | b[block k] == a[block k moved one column up] << 2.  first_lut[flags] = seed_first_slow.
// seed_flags_slow is the definition; seed_flags finds the zero fields of the three difference words at once (a field x is
// non-zero iff ((x_low + low_ones) | x) has its top bit set, exact per field and free of carries across fields).
BDG_HD uint32_t seed_flags_slow(const SeedScheme& s, uint32_t a, uint32_t b)
{
    const uint32_t x0 = a ^ b, xa = a ^ (b >> 2), xb = b ^ (a >> 2);
    uint32_t f = 0;
    for (int k = 0; k < s.nblocks; k++) {
        const uint32_t m = low_mask(s.bn[k]) << s.blo[k];
        f |= (((x0 & m) == 0 ? 1u : 0u) | ((xa & m) == 0 ? 2u : 0u) | ((xb & m) == 0 ? 4u : 0u)) << (3 * k);
    }
    return f;
}

BDG_HD uint32_t seed_flags(const SeedScheme& s, uint32_t a, uint32_t b)
{
    const uint32_t x0 = a ^ b, xa = a ^ (b >> 2), xb = b ^ (a >> 2);
    const uint32_t HI = s.hi_mask, LM = s.lo_mask;
    const uint32_t z0 = ~(((x0 & LM) + LM) | x0) & HI;        // top bit of every block whose field of x0 is zero
    const uint32_t za = ~(((xa & LM) + LM) | xa) & HI;
    const uint32_t zb = ~(((xb & LM) + LM) | xb) & HI;
    const uint32_t z = (z0 >> 2) | (za >> 1) | zb;             // three flags below / at the top bit of every block (blocks have >= 4 bits)
    uint32_t f = 0;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int k = 0; k < SEED_MAX_BLOCKS; k++) f |= (z & s.fmask[k]) >> s.fnet[k];      // block k's flags move down to bit 3k (fmask 0: no such block)
    return f;
}

// ---- the per-pair filter of the t = 2 join and the hand-over that knows it --------------------------------------------
// join_kernel<2, RS, SHF> tests a (row x, column y) pair of equal keys with
//   SHF (a shifted condition): at most two columns of x[0:15] mismatch y on both diagonals 0 and +1 - the frame of the
//                              condition's own diagonals (x[block] == y[block + d], d in {0, 1});
//   symmetric condition:       the same on {0, +1} OR on {0, -1}: either side, since the buckets hold the pair in no fixed order.
// yP = y >> 2, yM = y << 2 (yM unused by SHF).  A pair with D <= 2 always passes the symmetric test; it passes the shifted one
// under the labelling whose diagonals are >= 0, which is the labelling in which it meets a shifted condition.
template <bool SHF>
BDG_HD bool join2_quick(uint32_t x, uint32_t y, uint32_t yP, uint32_t yM, uint32_t one, uint32_t mone)
{
    if constexpr (SHF) return marks_le2(side_marks(x, y, yP), one, mone);
    else return marks_le2(side_marks(x, y, yP), one, mone) | marks_le2(side_marks(x, y, yM), one, mone);
}

// The two side bits of a pair a < b: bit 0 = the row test of a shifted condition with (row, column) = (a, b) passes, bit 1 = the
// same with (b, a).  The very function of the kernel's filter, so that the hand-over never names a pass whose filter dropped the pair.
BDG_HD uint32_t seed_side_bits(uint32_t a, uint32_t b)
{
    return (join2_quick<true>(a, b, b >> 2, 0u, 1u, 0xFFFFFFFFu) ? 1u : 0u) | (join2_quick<true>(b, a, a >> 2, 0u, 1u, 0xFFFFFFFFu) ? 2u : 0u);
}

// The hand-over of the t = 2 join: the first (condition, orientation) in table order that the pair meets AND whose kernel filter
// passes it - symmetric: always (the table is read for pairs with D <= 2 only, and they all pass); shifted, o = 0: side bit 0;
// shifted, o = 1: side bit 1.  Every pair with D <= 2 has exactly one owner: its labelling with diagonals >= 0 meets some
// condition, and the one-sided test passes in that labelling.  The definition; the kernels read the table below at
// seed_flags | seed_side_bits << nflags.
BDG_HD int seed_first_sides_slow(const SeedScheme& s, uint32_t a, uint32_t b)
{
    const uint32_t sides = seed_side_bits(a, b);
    for (int c = 0; c < s.nconds; c++) {
        if (seed_pred(s, c, a, b) && (s.cond[c].self || (sides & 1u))) return 2 * c;
        if (!s.cond[c].self && seed_pred(s, c, b, a) && (sides & 2u)) return 2 * c + 1;
    }
    return SEED_NONE;
}

// ---- host side: table of conditions, sort forms, hand-over table -------------------------------------------------
// blocks: number of bases of every block (sum 15).  Returns false if the layout does not fit the limits.
inline bool seed_scheme_build(SeedScheme& s, const int* bases, int nblocks)
{
    s = SeedScheme{};
    if (nblocks < 3 || nblocks > SEED_MAX_BLOCKS || nblocks - 2 > SEED_MAX_FIELDS) return false;
    int col = 0;
    for (int k = 0; k < nblocks; k++) { s.blo[k] = (uint8_t)(2 * col); s.bn[k] = (uint8_t)(2 * bases[k]); col += bases[k]; }
    if (col != 15) return false;
    s.nblocks = nblocks;
    s.nflags = 3 * nblocks;
    for (int k = 0; k < nblocks; k++) {
        if (bases[k] < 2) return false;                    // the flag extraction wants >= 4 bits per block
        s.hi_mask |= 1u << (s.blo[k] + s.bn[k] - 1);
        s.lo_mask |= low_mask(s.bn[k] - 1) << s.blo[k];
        s.fmask[k] = 7u << (s.blo[k] + s.bn[k] - 3);
        s.fnet[k] = (uint32_t)(s.blo[k] + s.bn[k] - 3 - 3 * k);
    }
    const int nf = nblocks - 2;
    {                                                      // block set by block set: its symmetric condition, then the shifted ones
        for (uint32_t sub = 0; sub < (1u << nblocks); sub++) {
            if (popc(sub) != nf) continue;
            int blk[SEED_MAX_FIELDS], q = 0;
            for (int k = 0; k < nblocks; k++) if (sub & (1u << k)) blk[q++] = k;
            s.set_first[s.nsets++] = (uint16_t)s.nconds;        // every set has its symmetric condition, so it is never empty
            for (uint32_t dm = 0; dm < (1u << nf); dm++) {      // bit f: diagonal of field f
                bool ok = true;
                if (blk[0] == 0 && (dm & 1u)) ok = false;                                     // block 0 sits on diagonal 0
                for (int f = 0; f + 1 < nf && ok; f++)
                    if (blk[f + 1] == blk[f] + 1 && (((dm >> f) ^ (dm >> (f + 1))) & 1u)) ok = false;   // neighbours share the diagonal
                if (!ok) continue;
                if (s.nconds >= SEED_MAX_CONDS) return false;
                SeedCond& c = s.cond[s.nconds];
                c.nf = (uint8_t)nf;
                c.self = dm == 0;
                SeedKey& ka = s.ka[s.nconds];
                SeedKey& kb = s.kb[s.nconds];
                ka.nf = kb.nf = (uint8_t)nf;
                int bits = 0;
                for (int f = 0; f < nf; f++) {
                    c.blk[f] = (uint8_t)blk[f];
                    c.d[f] = (uint8_t)((dm >> f) & 1u);
                    ka.lo[f] = s.blo[blk[f]]; kb.lo[f] = (uint8_t)(s.blo[blk[f]] + 2 * c.d[f]);
                    ka.n[f] = kb.n[f] = s.bn[blk[f]];
                    ka.at[f] = kb.at[f] = (uint8_t)bits;
                    ka.mask[f] = kb.mask[f] = low_mask(s.bn[blk[f]]);
                    bits += s.bn[blk[f]];
                }
                ka.key_bits = kb.key_bits = (uint8_t)bits;
                c.row_sort = (uint8_t)s.nconds;
                for (int e = 0; e < s.nconds; e++) {
                    bool same = true;
                    for (int f = 0; f < nf; f++) same = same && s.cond[e].blk[f] == c.blk[f];
                    if (same) { c.row_sort = s.cond[e].row_sort; break; }
                }
                s.nconds++;
            }
        }
    }
    s.set_first[s.nsets] = (uint16_t)s.nconds;
    for (int c = 0; c < s.nconds; c++) s.nself += s.cond[c].self;
    return true;
}

// lut: 1 << s.nflags entries
inline void seed_lut_build(const SeedScheme& s, uint8_t* lut)
{
    for (uint32_t f = 0; f < (1u << s.nflags); f++) {
        uint8_t first = SEED_NONE;
        for (int c = 0; c < s.nconds && first == SEED_NONE; c++) {
            for (int o = 0; o < (s.cond[c].self ? 1 : 2) && first == SEED_NONE; o++) {
                bool all = true;
                for (int k = 0; k < s.cond[c].nf; k++) {
                    const int b = s.cond[c].blk[k];
                    const int bit = 3 * b + (s.cond[c].d[k] == 0 ? 0 : (o == 0 ? 1 : 2));
                    all = all && ((f >> bit) & 1u);
                }
                if (all) first = (uint8_t)(2 * c + o);
            }
        }
        lut[f] = first;
    }
}

// lut: 1 << (s.nflags + 2) entries, lut[flags | sides << nflags] = seed_first_sides_slow.  One walk of the conditions per flag
// word fills its four side combinations.
inline void seed_lut_build_sides(const SeedScheme& s, uint8_t* lut)
{
    const uint32_t nf = 1u << s.nflags;
    for (uint32_t f = 0; f < nf; f++) {
        uint8_t first[4] = {SEED_NONE, SEED_NONE, SEED_NONE, SEED_NONE};
        int open = 4;
        for (int c = 0; c < s.nconds && open; c++) {
            for (int o = 0; o < (s.cond[c].self ? 1 : 2); o++) {
                bool all = true;
                for (int k = 0; k < s.cond[c].nf; k++) {
                    const int b = s.cond[c].blk[k];
                    const int bit = 3 * b + (s.cond[c].d[k] == 0 ? 0 : (o == 0 ? 1 : 2));
                    all = all && ((f >> bit) & 1u);
                }
                if (!all) continue;
                for (uint32_t sd = 0; sd < 4; sd++)
                    if (first[sd] == SEED_NONE && (s.cond[c].self || ((sd >> o) & 1u))) { first[sd] = (uint8_t)(2 * c + o); open--; }
            }
        }
        for (uint32_t sd = 0; sd < 4; sd++) lut[f | sd << s.nflags] = first[sd];
    }
}

}  // namespace bdg
