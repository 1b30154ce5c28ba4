// bdg_seed3.cuh -- multi-block seeds for the t = 3 edge construction by sort-merge joins (bdg_join.cuh).
//
// What is searched (reference index.py:77-93 + barcode_graph.py:233-249): pairs a < b with D(a,b) <= 3 and S(a,b) >= 4
// (T(3) = 4, the same candidate threshold as t = 2).  The necessary condition extends the t = 2 one of bdg_seed.cuh:
//   * cut a[0:15] into B blocks (column 15 is left out: the truncated variants of D drop it for free);
//   * an edit script of <= 3 operations touches <= 3 blocks (an insertion in front of a[i] is charged to the block holding
//     a[i]), so >= B-3 blocks are untouched and each of them equals a stretch of b on one diagonal d = #insertions -
//     #deletions in front of it;
//   * the three alignments behind D end at net shift -1, 0 or +1, so every untouched block has d in [-2, +2];
//   * unlike t = 2 both signs occur in one pair (0 -> +1 -> 0 -> -1 takes three indels), so there is no "all diagonals >= 0
//     under one labelling": every condition keeps its signs and is joined in both value orders.
// A condition = B-3 blocks u_1 < ... < u_m with a diagonal d_i in [-2, 2] each, kept iff
//   * d_1 = 0 if u_1 = 0 (nothing in front of block 0);
//   * adjacent blocks (u_{i+1} = u_i + 1) share their diagonal (nothing between them can change it);
//   * the indels it implies fit the budget: |d_1| + sum |d_{i+1} - d_i| + max(0, |d_m| - 1) <= 3;
//   * no block is shifted outside b's 16 columns.
//   B = 5 (3 x 5 bases): 82 conditions (10 symmetric);  B = 6 (3,3,3,2,2,2): 242 (20);  B = 7 (3,2,2,2,2,2,2): 539 (35).
// As at t = 2 a condition is a plain key equality "these fields of x equal those fields of y" (SeedKey of bdg_seed.cuh, keys of
// <= 20 bits), so the counting sort of bdg_join.cuh buckets both sides unchanged.
//
// Hand-over: a pair that meets several conditions is emitted by the FIRST (condition, orientation) in table order
// (seed3_first_slow is the definition).  The t = 2 table over all block-match flags does not scale (5 diagonals x 7 blocks =
// 35 flag bits per orientation), so seed3_first walks the table instead, cheaply: the pair's match flags of every (block,
// diagonal) are found for both orientations with the zero-field trick of bdg_seed.cuh (seed3_flags, one 64-bit word each), a
// condition is met iff its required flags are all set, and a whole block set is skipped unless each of its blocks matches on
// some diagonal.  A close pair matches few blocks off its own diagonals, so the walk visits a handful of sets in full.
//
// Everything is __host__ __device__: tests/test_seed3_host.py compiles this header with g++ and checks necessity against the
// oracle's distances, seed3_first against the definition, and the emulated passes against the oracle's edge set.
#pragma once
#include "bdg_seed.cuh"

namespace bdg {

constexpr int SEED3_MAX_BLOCKS = 7;
constexpr int SEED3_MAX_CONDS = 640;
constexpr int SEED3_MAX_SETS = 35;                 // C(7, 4): block sets of the largest layout
constexpr int SEED3_NONE = 0xFFFF;

struct Seed3Cond {
    uint8_t nf;                       // number of blocks in the condition (B - 3)
    uint8_t blk[SEED_MAX_FIELDS];     // ascending
    int8_t d[SEED_MAX_FIELDS];        // diagonal of each block, -2..2 (x[block] == y[block columns + d])
    uint8_t self;                     // all diagonals 0
    uint16_t set;                     // block set: the conditions of a set follow one another, the symmetric one first
};

struct Seed3Scheme {
    int nblocks;
    uint8_t blo[SEED3_MAX_BLOCKS], bn[SEED3_MAX_BLOCKS];   // first bit / number of bits of every block
    int nconds, nself, nsets;
    Seed3Cond cond[SEED3_MAX_CONDS];
    SeedKey ka[SEED3_MAX_CONDS], kb[SEED3_MAX_CONDS];       // join key of the row side (fields of x) / column side (fields of y)
    uint64_t need[SEED3_MAX_CONDS];                         // flags of seed3_flags the condition requires
    uint16_t set_first[SEED3_MAX_SETS + 1];                 // conditions of set s: set_first[s] .. set_first[s + 1] - 1
    uint32_t set_hi[SEED3_MAX_SETS];                        // top bit of every block of set s
    uint32_t hi_mask, lo_mask;                              // top bit of every block / the other bits of the blocks
};

BDG_HD uint32_t shift_diag(uint32_t y, int d) { return d >= 0 ? y >> (2 * d) : y << (-2 * d); }   // y moved so that y[i + d] sits at column i

// x[fields of condition c] == y[the same fields moved by their diagonals]
BDG_HD bool seed3_pred(const Seed3Scheme& s, int c, uint32_t x, uint32_t y) { return seed_key(x, s.ka[c]) == seed_key(y, s.kb[c]); }

// first (condition, orientation) the pair meets, as 2 * c + o (o = 0: (x, y) = (a, b); o = 1: (x, y) = (b, a)), by the
// definition; SEED3_NONE if none.
BDG_HD int seed3_first_slow(const Seed3Scheme& s, uint32_t a, uint32_t b)
{
    for (int c = 0; c < s.nconds; c++) {
        if (seed3_pred(s, c, a, b)) return 2 * c;
        if (!s.cond[c].self && seed3_pred(s, c, b, a)) return 2 * c + 1;
    }
    return SEED3_NONE;
}

// Block-match flags of (x, y): block k matches y on diagonal d (x[block k] == y[block k columns + d]) <=> bit (top bit of block
// k) - (d + 2) for d = -2..1, bit 32 + (top bit of block k) for d = 2.  Blocks have >= 4 bits, so the four low flags stay inside
// the block.  *any: the top bit of every block that matches on some diagonal.
BDG_HD uint64_t seed3_flags(const Seed3Scheme& s, uint32_t x, uint32_t y, uint32_t* any)
{
    const uint32_t HI = s.hi_mask, LM = s.lo_mask;
    uint32_t z[5];
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int d = -2; d <= 2; d++) {
        const uint32_t X = x ^ shift_diag(y, d);
        z[d + 2] = ~(((X & LM) + LM) | X) & HI;              // top bit of every block whose field of X is zero
    }
    *any = z[0] | z[1] | z[2] | z[3] | z[4];
    return (uint64_t)(z[0] | (z[1] >> 1) | (z[2] >> 2) | (z[3] >> 3)) | ((uint64_t)z[4] << 32);
}

// seed3_first_slow by the flags: the form the kernel uses
BDG_HD int seed3_first(const Seed3Scheme& s, uint32_t a, uint32_t b)
{
    uint32_t any0 = 0, any1 = 0;
    const uint64_t f0 = seed3_flags(s, a, b, &any0), f1 = seed3_flags(s, b, a, &any1);
    for (int k = 0; k < s.nsets; k++) {
        const uint32_t h = s.set_hi[k];
        const bool p0 = (any0 & h) == h, p1 = (any1 & h) == h;
        if (!p0 && !p1) continue;
        for (int c = s.set_first[k]; c < s.set_first[k + 1]; c++) {
            const uint64_t n = s.need[c];
            if (p0 && (f0 & n) == n) return 2 * c;
            if (p1 && !s.cond[c].self && (f1 & n) == n) return 2 * c + 1;
        }
    }
    return SEED3_NONE;
}

// The kernel's quick test: with <= 3 operations every column 0..14 of a is matched on one of the diagonals -2..2 or consumed by
// an operation, so more than three columns that mismatch on all five prove D > 3 (quick_pass_any with k = 2; the bases
// shifted in at the ends count as possible matches here, which only weakens the test).  Marks on the odd bits as in quick_marks.
BDG_HD uint32_t quick3_marks(uint32_t a, uint32_t b0, uint32_t bP, uint32_t bM)
{
    const uint32_t xp2 = a ^ (bP >> 2), xm2 = a ^ (bM << 2);
    return quick_marks(a, b0, bP, bM) & (xp2 | (xp2 << 1)) & (xm2 | (xm2 << 1));
}
BDG_HD bool quick3_pass(uint32_t a, uint32_t b)
{
    uint32_t u = quick3_marks(a, b, b >> 2, b << 2);
    for (int i = 0; i < 3; i++) u &= u - 1;      // drop the three lowest marks
    return u == 0;
}

// ---- host side: table of conditions -----------------------------------------------------------------------------------
// bases: number of bases of every block (sum 15, each >= 2).  Returns false if the layout does not fit the limits.
inline bool seed3_scheme_build(Seed3Scheme& s, const int* bases, int nblocks)
{
    s = Seed3Scheme{};
    if (nblocks < 4 || nblocks > SEED3_MAX_BLOCKS || nblocks - 3 > SEED_MAX_FIELDS) return false;
    int col = 0, first_col[SEED3_MAX_BLOCKS];
    for (int k = 0; k < nblocks; k++) {
        if (bases[k] < 2) return false;                    // the flag extraction wants >= 4 bits per block
        first_col[k] = col;
        s.blo[k] = (uint8_t)(2 * col); s.bn[k] = (uint8_t)(2 * bases[k]); col += bases[k];
    }
    if (col != 15) return false;
    s.nblocks = nblocks;
    for (int k = 0; k < nblocks; k++) {
        s.hi_mask |= 1u << (s.blo[k] + s.bn[k] - 1);
        s.lo_mask |= low_mask(s.bn[k] - 1) << s.blo[k];
    }
    const int nf = nblocks - 3;
    static const int DIAG[5] = {0, 1, -1, 2, -2};         // digit -> diagonal: the all-zero (symmetric) vector comes first
    int n_vec = 1;
    for (int f = 0; f < nf; f++) n_vec *= 5;
    for (uint32_t sub = 0; sub < (1u << nblocks); sub++) {
        if (popc(sub) != nf) continue;
        int blk[SEED_MAX_FIELDS], q = 0;
        for (int k = 0; k < nblocks; k++) if (sub & (1u << k)) blk[q++] = k;
        if (s.nsets >= SEED3_MAX_SETS) return false;
        const int set = s.nsets++;
        s.set_first[set] = (uint16_t)s.nconds;
        for (int f = 0; f < nf; f++) s.set_hi[set] |= 1u << (s.blo[blk[f]] + s.bn[blk[f]] - 1);
        for (int v = 0; v < n_vec; v++) {
            int d[SEED_MAX_FIELDS];
            for (int f = 0, r = v; f < nf; f++, r /= 5) d[f] = DIAG[r % 5];
            bool ok = !(blk[0] == 0 && d[0] != 0);                                         // block 0 sits on diagonal 0
            int cost = d[0] < 0 ? -d[0] : d[0];
            for (int f = 0; f < nf && ok; f++) {
                const int c0 = first_col[blk[f]] + d[f], c1 = first_col[blk[f]] + bases[blk[f]] - 1 + d[f];
                if (c0 < 0 || c1 > 15) ok = false;                                             // inside b's 16 columns
                if (f + 1 < nf) {
                    const int step = d[f + 1] - d[f];
                    if (blk[f + 1] == blk[f] + 1 && step != 0) ok = false;                     // neighbours share the diagonal
                    cost += step < 0 ? -step : step;
                }
            }
            const int last = d[nf - 1] < 0 ? -d[nf - 1] : d[nf - 1];
            cost += last > 1 ? last - 1 : 0;
            if (!ok || cost > 3) continue;
            if (s.nconds >= SEED3_MAX_CONDS) return false;
            Seed3Cond& c = s.cond[s.nconds];
            SeedKey& ka = s.ka[s.nconds];
            SeedKey& kb = s.kb[s.nconds];
            c.nf = (uint8_t)nf;
            c.set = (uint16_t)set;
            c.self = 1;
            ka.nf = kb.nf = (uint8_t)nf;
            int bits = 0;
            uint64_t need = 0;
            for (int f = 0; f < nf; f++) {
                const int b = blk[f], top = s.blo[b] + s.bn[b] - 1;
                c.blk[f] = (uint8_t)b;
                c.d[f] = (int8_t)d[f];
                if (d[f] != 0) c.self = 0;
                ka.lo[f] = s.blo[b]; kb.lo[f] = (uint8_t)(s.blo[b] + 2 * d[f]);
                ka.n[f] = kb.n[f] = s.bn[b];
                ka.at[f] = kb.at[f] = (uint8_t)bits;
                ka.mask[f] = kb.mask[f] = low_mask(s.bn[b]);
                bits += s.bn[b];
                need |= d[f] == 2 ? (1ull << (32 + top)) : (1ull << (top - (d[f] + 2)));
            }
            if (bits > 20) return false;                   // one digit of the counting sort
            ka.key_bits = kb.key_bits = (uint8_t)bits;
            s.need[s.nconds] = need;
            s.nself += c.self;
            s.nconds++;
        }
    }
    s.set_first[s.nsets] = (uint16_t)s.nconds;
    return true;
}

}  // namespace bdg
