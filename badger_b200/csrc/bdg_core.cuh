// bdg_core.cuh -- per-pair arithmetic of the barcode hot path on packed 16-mers.
//
// A barcode is a uint32 in the reference's own packing (reference common.py:21-25): base i occupies
// bits 2i..2i+1, A0 C1 G2 T3.  Everything here is integer bit arithmetic on those words.
//
// The functions are __host__ __device__ so that tests/test_core_host.py can compile this very header
// with g++ and check every function against the CPU oracle on millions of pairs without a GPU.  The
// product only ever calls them from CUDA kernels (bdg_kernels.cu); there is no CPU execution path.
//
// Reference semantics restated (file:line in /root/reference):
//   D(a,b) = min(ed(a,b), ed(a[:-1],b), ed(a,b[:-1]))          barcode_graph.py:96, :243
//   S(a,b) = #{(p,q) in [0,10]^2 : 6mer_a[p] == 6mer_b[q]}      index.py:29-35, :77-93
//   T(t)   = 16-6+1-6t, replaced by 4 when <= 0                 index.py:19-24
//   edge(a,b) <=> a<b, S >= T(t), D <= t ; stored distance = D  barcode_graph.py:233-249
//   plain ed(q,c) for --high_sens post-processing               barcode_graph.py:379
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define BDG_HD __host__ __device__ __forceinline__
#else
#define BDG_HD static inline
#endif

namespace bdg {

constexpr uint32_t EVEN = 0x55555555u;   // one marker bit per base (bit 2i)
constexpr uint32_t ODD = 0xAAAAAAAAu;

BDG_HD int popc(uint32_t x)
{
#if defined(__CUDA_ARCH__)
    return __popc(x);
#else
    return __builtin_popcount(x);
#endif
}

// T(t): index.py:22-24
BDG_HD int qgram_threshold(int t)
{
    int T = 16 - 6 + 1 - 6 * t;
    return T <= 0 ? 4 : T;
}

// Mismatch marks of two aligned words: bit 2i set <=> base i differs.
BDG_HD uint32_t mism(uint32_t a, uint32_t b)
{
    uint32_t x = a ^ b;
    return (x | (x >> 1)) & EVEN;
}

// ---------------------------------------------------------------------------------------------
// Stage-1 prefilters: cheap NECESSARY conditions for D(a,b) <= t.  A reject proves D > t.
//
// Why only the diagonals -1, 0, +1 matter for t <= 2: the three alignments behind D have length
// differences 0, +1, -1, and an edit script of <= 2 operations with that net length change can hold
// at most one insertion and one deletion, so no aligned column is ever more than one base off the main
// diagonal.  Every script cuts a[0:15] with at most two "events" (a substituted column, a removed base
// or a diagonal change), so of any three disjoint blocks of a[0:15] one is untouched and matches b
// exactly on diagonal -1, 0 or +1 (pigeonhole).
//
//   t = 2: blocks a[0:5], a[5:10], a[10:15] = bit fields 0-9, 10-19, 20-29 against b, b>>2, b<<2.
//   t = 1: one event, two blocks: a[0:8] / a[8:16] on diagonal 0, a[8:15] on +1, a[9:16] on -1.
//
// "some field of x is zero" is evaluated for all fields of a word at once with the classic
// (x - ones) & ~x & highs test, which is exact as a whole-word predicate.
// ---------------------------------------------------------------------------------------------
constexpr uint32_t F10_ONES = (1u << 0) | (1u << 10) | (1u << 20);
constexpr uint32_t F10_HIGH = (1u << 9) | (1u << 19) | (1u << 29);
constexpr uint32_t F16_ONES = 0x00010001u;
constexpr uint32_t F16_HIGH = 0x80008000u;

// second word of the t=1 test: low half = a[8:15] (for diagonal +1), high half = a[9:16] (diagonal -1)
BDG_HD uint32_t t1_word_a(uint32_t a) { return ((a >> 16) & 0x3FFFu) | ((a >> 18) << 16); }
// matching word of b: low half = b[9:16], high half = b[8:15]
BDG_HD uint32_t t1_word_b(uint32_t b) { return (b >> 18) | (((b >> 16) & 0x3FFFu) << 16); }

BDG_HD uint32_t zero_field_marks(uint32_t x, uint32_t ones) { return (x - ones) & ~x; }

BDG_HD bool prefilter_t1(uint32_t a, uint32_t b)
{
    uint32_t m = zero_field_marks(a ^ b, F16_ONES) | zero_field_marks(t1_word_a(a) ^ t1_word_b(b), F16_ONES);
    return (m & F16_HIGH) != 0;
}

BDG_HD bool prefilter_t2(uint32_t a, uint32_t b)
{
    uint32_t m = zero_field_marks(a ^ b, F10_ONES) | zero_field_marks(a ^ (b >> 2), F10_ONES) |
                 zero_field_marks(a ^ (b << 2), F10_ONES);
    return (m & F10_HIGH) != 0;
}

// ---------------------------------------------------------------------------------------------
// The prefilters split in two for the tiled edge kernel (bdg_edges.cuh).  The barcode array is SORTED, so
// inside a tile (a run of consecutive rows x a run of consecutive columns) the high bits of a and of b
// barely move.  Conditions that compare the TOP block of a with (a shift of) the top of b ("top" part) can
// therefore be excluded for a whole tile from the first/last element of its rows and columns
// (tX_top_possible); only the remaining conditions ("light" part) have to be evaluated pair by pair.
//
// Which conditions are needed (tighter than the 9/4 fields tested above): an insertion in front of a[i]
// is charged to the block holding a[i], so every operation touches one block, and an untouched block sits
// on diagonal (#insertions - #deletions before it).  Block 0 has nothing before it: diagonal 0 only.
//   t = 1, blocks a[0:8] | a[8:16]:   light  a[0:8]==b[0:8]   (kernel compares 15 of its 16 bits)
//                                     top    a[8:16]==b[8:16], a[8:15]==b[9:16], a[9:16]==b[8:15]
//   t = 2, blocks a[0:5] | a[5:10] | a[10:15]:
//                                     light  a[0:5]==b[0:5], a[5:10]==b[5:10], a[5:10]==b[6:11], a[5:10]==b[4:9]
//                                     top    a[10:15]==b[10:15], a[10:15]==b[11:16], a[10:15]==b[9:14]
// tests/test_core_host.py checks  D <= t  =>  light || top  on the oracle's distances, in both frames.
// ---------------------------------------------------------------------------------------------
BDG_HD bool t1_light(uint32_t a, uint32_t b) { return ((a ^ b) & 0x7FFFu) == 0; }

BDG_HD bool t1_top(uint32_t a, uint32_t b)
{
    return (a >> 16) == (b >> 16) || ((a >> 16) & 0x3FFFu) == (b >> 18) || (a >> 18) == ((b >> 16) & 0x3FFFu);
}

// t=2 light test words: two 10-bit fields in the two 16-bit lanes, bit 10 of each lane is a guard position
//   word A:  lane0 = block 0, lane1 = block 1                 (diagonal 0)
//   word B:  a: block 1 in both lanes;  b: lane0 = b[6:11] (diagonal +1), lane1 = b[4:9] (diagonal -1)
BDG_HD uint32_t t2_word_aA(uint32_t a) { return (a & 0x3FFu) | (((a >> 10) & 0x3FFu) << 16); }
BDG_HD uint32_t t2_word_aB(uint32_t a) { return ((a >> 10) & 0x3FFu) * 0x00010001u; }
BDG_HD uint32_t t2_word_bA(uint32_t b) { return t2_word_aA(b); }
BDG_HD uint32_t t2_word_bB(uint32_t b) { return ((b >> 12) & 0x3FFu) | (((b >> 8) & 0x3FFu) << 16); }
constexpr uint32_t T2_GUARD = 0x04000400u;

BDG_HD bool t2_light(uint32_t a, uint32_t b)
{
    // G - x keeps the guard bit of a lane iff the lane's field of x is zero (x < 2^10 per lane, no borrow across lanes)
    const uint32_t yA = T2_GUARD - (t2_word_aA(a) ^ t2_word_bA(b));
    const uint32_t yB = T2_GUARD - (t2_word_aB(a) ^ t2_word_bB(b));
    return ((yA | yB) & T2_GUARD) != 0;
}

BDG_HD bool t2_top(uint32_t a, uint32_t b)
{
    const uint32_t f = (a >> 20) & 0x3FFu;
    return f == ((b >> 20) & 0x3FFu) || f == (b >> 22) || f == ((b >> 18) & 0x3FFu);
}

// Values of the field v[x : x+len) over all v in [lo, hi]: v >> x runs through consecutive integers, so the field
// runs through a CYCLIC interval of the field's range: start = field(lo), length = (hi>>x) - (lo>>x) + 1, capped
// at the whole range.  Two such intervals meet iff either start lies inside the other one.
BDG_HD bool fields_may_meet(uint32_t alo, uint32_t ahi, int xa, uint32_t blo, uint32_t bhi, int xb, int len)
{
    const uint32_t mask = (1u << len) - 1u;          // len <= 16 here
    const uint32_t sa = (alo >> xa) & mask, sb = (blo >> xb) & mask;
    const uint32_t la = (ahi >> xa) - (alo >> xa) + 1u, lb = (bhi >> xb) - (blo >> xb) + 1u;
    return ((sb - sa) & mask) < la || ((sa - sb) & mask) < lb;
}

// Can ANY pair (a in [alo,ahi], b in [blo,bhi]) satisfy a top condition?  false => the whole tile skips them.
BDG_HD bool t1_top_possible(uint32_t alo, uint32_t ahi, uint32_t blo, uint32_t bhi)
{
    return fields_may_meet(alo, ahi, 16, blo, bhi, 16, 16) || fields_may_meet(alo, ahi, 16, blo, bhi, 18, 14) ||
           fields_may_meet(alo, ahi, 18, blo, bhi, 16, 14);
}

BDG_HD bool t2_top_possible(uint32_t alo, uint32_t ahi, uint32_t blo, uint32_t bhi)
{
    return fields_may_meet(alo, ahi, 20, blo, bhi, 20, 10) || fields_may_meet(alo, ahi, 20, blo, bhi, 22, 10) ||
           fields_may_meet(alo, ahi, 20, blo, bhi, 18, 10);
}

// ---------------------------------------------------------------------------------------------
// Multi-pass ("sparse") form of the same prefilter.  Every condition above compares a block of a with a
// block of b.  Sorting the barcodes by a ROTATED key puts any chosen block on top, and then that block's
// conditions can be excluded tile by tile exactly like the "top" part above.  With one pass per block no
// condition is left that needs a per-pair test over the whole matrix: pass p scans (row group x column
// sub-tile) intervals of the array sorted by rotl(key, rot_p) and evaluates its own conditions only inside
// the few tiles whose intervals meet.
//   t = 1:  pass 0  rot  0   a[8:16]==b[8:16], a[8:15]==b[9:16], a[9:16]==b[8:15]   (t1_top, closed under swap)
//           pass 1  rot 16   a[0:8]==b[0:8]
//   t = 2:  pass 0  rot  0   block 2 on diagonals 0, +1, -1, both orientations          (t2_blk3)
//           pass 1  rot 10   block 1 on diagonals 0, +1, -1, both orientations          (t2_blk3 on rotated words)
//           pass 2  rot 20   block 0 on diagonal 0                                      (t2_blk1 on rotated words)
// The predicates are orientation-free (they hold for (x,y) iff for (y,x)), so a pair is found no matter
// which of the two comes first in the rotated order.  A pair that satisfies the predicates of several
// passes is emitted by the FIRST of them only (pass_pred of the earlier passes is re-evaluated on the
// candidate), which keeps the edge list duplicate-free without any merge step.
// ---------------------------------------------------------------------------------------------
BDG_HD uint32_t rotl32(uint32_t v, int r) { return r ? ((v << r) | (v >> (32 - r))) : v; }
BDG_HD uint32_t rotr32(uint32_t v, int r) { return r ? ((v >> r) | (v << (32 - r))) : v; }

BDG_HD bool t2_blk3(uint32_t x, uint32_t y)   // words rotated so that the block sits in bits 20..29
{
    const uint32_t fx = (x >> 20) & 0x3FFu, fy = (y >> 20) & 0x3FFu;
    return fx == fy || fx == (y >> 22) || fx == ((y >> 18) & 0x3FFu) || fy == (x >> 22) || fy == ((x >> 18) & 0x3FFu);
}
BDG_HD bool t2_blk1(uint32_t x, uint32_t y) { return (((x ^ y) >> 20) & 0x3FFu) == 0; }

// Per-pair test of the sparse passes inside a surviving tile: NOT the pass predicate (that is re-checked on
// the few survivors, for the duplicate-free hand-over between passes) but the stronger necessary condition
// "at most t columns of a[0:15] mismatch on all three diagonals" (see dist_small's quick reject): with <= t
// operations every other column is matched on diagonal 0, +1 or -1.  Marks live on the ODD bits here
// (x | x<<1), so the shift is a multiply by two on the FMA pipe.  bP = b >> 2, bM = b << 2.
constexpr uint32_t QUICK_VALID = 0x2AAAAAAAu;   // columns 0..14, odd bits
BDG_HD uint32_t quick_marks(uint32_t a, uint32_t b0, uint32_t bP, uint32_t bM)
{
    const uint32_t x0 = a ^ b0, xp = a ^ bP, xm = a ^ bM;
    return (x0 | (x0 << 1)) & (xp | (xp << 1)) & (xm | (xm << 1)) & QUICK_VALID;
}
// One diagonal side of the same test: marks of the columns 0..14 of x that match y neither on diagonal 0 (yd = y) nor on the
// one shifted word ys (y >> 2: x[i] vs y[i + 1]).  Column 15 is left out and column 14 meets the zero shifted in at the top,
// exactly as in quick_marks.  A script of <= 2 operations keeps its columns on {0, +1} or on {0, -1} (bdg_seed.cuh), so under
// one labelling of a pair with D <= 2 at most two marks of side_marks(p, q, q >> 2) are set.
BDG_HD uint32_t side_marks(uint32_t x, uint32_t yd, uint32_t ys)
{
    const uint32_t x0 = x ^ yd, xs = x ^ ys;
    return (x0 | (x0 << 1)) & (xs | (xs << 1)) & QUICK_VALID;
}
// at most two marks: drop the two lowest, test for zero.  one / mone are 1 / -1 (the kernels pass them at run time, so that
// w * one + mone is an IMAD on the FMA pipe instead of an add on the ALU pipe)
BDG_HD bool marks_le2(uint32_t w, uint32_t one, uint32_t mone)
{
    w &= w * one + mone;
    w &= w * one + mone;
    return w == 0;
}
BDG_HD bool quick_pass(uint32_t a, uint32_t b, int t)
{
    uint32_t u = quick_marks(a, b, b >> 2, b << 2);
    for (int i = 0; i < t; i++) u &= u - 1;      // drop the t lowest marks
    return u == 0;
}

// The same idea for any threshold (dense kernel, t >= 3): with <= t operations and a length difference <= 1 no
// aligned column is more than k = (t+1)/2 bases off the main diagonal, so every column 0..14 of a is matched on one
// of the diagonals -k..k or consumed by an operation: more than t columns that mismatch on ALL of them prove D > t.
BDG_HD bool quick_pass_any(uint32_t a, uint32_t b, int t)
{
    const int k = (t + 1) / 2;
    const uint32_t x0 = a ^ b;
    uint32_t u = (x0 | (x0 << 1)) & QUICK_VALID;
    for (int s = 1; s <= k && s < 16 && u; s++) {
        const uint32_t xp = a ^ (b >> (2 * s));                 // a[i] vs b[i+s]: columns 16-s.. have no partner ...
        const uint32_t xm = a ^ (b << (2 * s));                 // a[i] vs b[i-s]: columns ..s-1 have no partner
        const uint32_t nop = ~(0xFFFFFFFFu >> (2 * s)), nom = ~(0xFFFFFFFFu << (2 * s));   // ... and count as mismatches there
        u &= ((xp | (xp << 1)) | nop) & ((xm | (xm << 1)) | nom);
    }
    for (int i = 0; i < t && u; i++) u &= u - 1;
    return u == 0;
}

constexpr int MAX_PASSES = 3;
BDG_HD int n_passes(int t) { return t == 1 ? 2 : (t == 2 ? 3 : 0); }
BDG_HD int pass_rot(int t, int p) { return t == 1 ? (p == 1 ? 16 : 0) : 10 * p; }

// predicate of pass p on ORIGINAL (unrotated) words
BDG_HD bool pass_pred(int t, int p, uint32_t x, uint32_t y)
{
    if (t == 1) return p == 0 ? t1_top(x, y) : ((x ^ y) & 0xFFFFu) == 0;
    if (p == 0) return t2_blk3(x, y);
    if (p == 1) return t2_blk3(rotl32(x, 10), rotl32(y, 10));
    return t2_blk1(rotl32(x, 20), rotl32(y, 20));
}

// the same predicate on words already rotated by pass_rot(t, p)
BDG_HD bool pass_pred_rot(int t, int p, uint32_t xr, uint32_t yr)
{
    if (t == 1) return p == 0 ? t1_top(xr, yr) : (xr >> 16) == (yr >> 16);
    return p == 2 ? t2_blk1(xr, yr) : t2_blk3(xr, yr);
}

// Can any (a in [alo,ahi], b in [blo,bhi]) - rotated keys of pass p - satisfy pass_pred_rot?
BDG_HD bool pass_possible(int t, int p, uint32_t alo, uint32_t ahi, uint32_t blo, uint32_t bhi)
{
    if (t == 1) {
        if (p == 0) return t1_top_possible(alo, ahi, blo, bhi);
        return fields_may_meet(alo, ahi, 16, blo, bhi, 16, 16);
    }
    if (p == 2) return fields_may_meet(alo, ahi, 20, blo, bhi, 20, 10);
    return fields_may_meet(alo, ahi, 20, blo, bhi, 20, 10) || fields_may_meet(alo, ahi, 20, blo, bhi, 22, 10) ||
           fields_may_meet(alo, ahi, 20, blo, bhi, 18, 10) || fields_may_meet(alo, ahi, 22, blo, bhi, 20, 10) ||
           fields_may_meet(alo, ahi, 18, blo, bhi, 20, 10);
}

// ---------------------------------------------------------------------------------------------
// Stage-2, exact for small distances: returns min(D(a,b), 3) for a != b, i.e. 1, 2, or 3 (= "3 or more").
// With plain_only it returns min(ed(a,b), 3) instead (no truncated variants; barcode_graph.py:379).
//
// Case analysis of all edit scripts of length <= 2 (see the block comment above):
//   ed(a,b):        <=2 substitutions                      -> popc(X0) <= 2
//                   1 deletion + 1 insertion, no mismatch  -> X0 clean outside [L,H], the middle clean on
//                                                             diagonal -1 (or +1), L/H = first/last mark of X0
//   ed(a[:15],b):   1 insertion in b + <=1 substitution    -> diagonal 0 before it, +1 after it
//   ed(a,b[:15]):   1 deletion from a + <=1 substitution   -> diagonal 0 before it, -1 after it
// X0 / XP / XM are the mismatch marks on diagonals 0 / +1 / -1 with out-of-range columns marked.
// ---------------------------------------------------------------------------------------------
// prefiltered: the caller's candidates already passed quick_marks' test (the join kernel), so the quick reject is left out -
// it only ever saves work, the case analysis behind it is exact on its own.
BDG_HD int dist_small(uint32_t a, uint32_t b, bool plain_only = false, bool prefiltered = false)
{
    const uint32_t X0 = mism(a, b);
    const int h = popc(X0);
    if (h == 0) return 0;                              // identical words (callers exclude this)
    const uint32_t XP = mism(a, b >> 2) | (1u << 30);  // a[i] vs b[i+1], i = 0..14; column 15 invalid
    const uint32_t XM = mism(a, b << 2) | 1u;          // a[i] vs b[i-1], i = 1..15; column 0 invalid
    // quick reject: with <= 2 operations every column 0..14 of a is either matched on diagonal 0, +1 or -1 or
    // consumed by an operation, so more than two columns that mismatch on all three diagonals prove D >= 3
    // (column 15 is left out: the truncated variants drop it for free).  Rejects ~90 % of the candidates.
    if (!prefiltered && popc(X0 & XP & XM & 0x15555555u) > 2) return 3;
    const uint32_t low1 = X0 & (0u - X0);              // first mismatch on the main diagonal (position L)
    const uint32_t ge1 = 0u - low1;                    // columns >= L (all bits from low1 upwards)
    const uint32_t gt1 = ge1 << 2;                     // columns >  L (marker bits; ge1 has both bits of a column set)
    int best = h <= 2 ? h : 3;
    if (h >= 2) {
        // one deletion + one insertion: the columns strictly between the events run on one side diagonal
        uint32_t s = X0;                               // smear downwards: all columns <= H
        s |= s >> 2; s |= s >> 4; s |= s >> 8; s |= s >> 16;
        const uint32_t leH = s;                        // marker bits of columns <= H (H = last mismatch)
        const uint32_t ltH = s >> 2;                   // columns < H
        const bool delins = (XM & gt1 & leH) == 0;     // a[L] removed, b gains a base after column H: XM clean on (L,H]
        const bool insdel = (XP & ge1 & ltH) == 0;     // b gains a base at L, a[H] removed:           XP clean on [L,H)
        if (delins || insdel) best = 2;
    }
    if (plain_only) return best;
    // truncated variants: one indel (free last base) + at most one substitution
    const uint32_t VALID15 = EVEN & 0x3FFFFFFFu;       // columns 0..14
    {
        // ed(a[:15], b): diagonal 0 on [0,p), diagonal +1 on [p,15)
        const uint32_t tailP = XP & ge1 & VALID15;     // p = L
        const int cP = popc(tailP);
        // ed(a, b[:15]): diagonal 0 on [0,p), a[p] removed, diagonal -1 on (p,16)
        const uint32_t tailM = XM & gt1;
        const int cM = popc(tailM);
        if (cP == 0 || cM == 0) return 1;
        if (cP == 1 || cM == 1) best = best < 2 ? best : 2;
        // or spend the substitution on the main diagonal: run through L up to the second mismatch L2
        const uint32_t X0b = X0 & (X0 - 1);            // X0 without its first mark
        const uint32_t low2 = X0b & (0u - X0b);
        const uint32_t ge2 = X0b ? (0u - low2) : 0u;   // columns >= L2 (none when X0 has a single mark)
        const uint32_t gt2 = ge2 << 2;
        if ((XP & ge2 & VALID15) == 0 || (XM & gt2) == 0) best = best < 2 ? best : 2;
    }
    return best;
}

// ---------------------------------------------------------------------------------------------
// Generic exact distances (any threshold): Myers' bit-vector algorithm for GLOBAL edit distance with the
// pattern a on the rows, run directly on the 2-bit-stride words (marker bit 2i = row i; the odd bits are
// fed as ones into the adder so carries ripple from row to row).  One pass yields all three distances of
// barcode_graph.py:243:  ed(a,b[:15]) = bottom-row score after column 15, ed(a,b) after column 16,
// ed(a[:15],b) = ed(a,b) minus the vertical delta of the last row in the last column.
// ---------------------------------------------------------------------------------------------
struct Dist3 { int full, a15, b15; };   // ed(a,b), ed(a[:15],b), ed(a,b[:15])

BDG_HD Dist3 myers3(uint32_t a, uint32_t b)
{
    uint32_t Pv = EVEN, Mv = 0;
    int score = 16, score15 = 16;
    const uint32_t TOP = 1u << 30;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int j = 0; j < 16; j++) {
        const uint32_t c = (b >> (2 * j)) & 3u;
        const uint32_t x = a ^ (c * EVEN);
        const uint32_t Eq = ~(x | (x >> 1)) & EVEN;
        const uint32_t Xv = Eq | Mv;
        const uint32_t Xh = ((((Eq & Pv) + (Pv | ODD)) ^ Pv) | Eq) & EVEN;
        uint32_t Ph = (Mv | ~(Xh | Pv)) & EVEN;
        uint32_t Mh = Pv & Xh;
        score += (Ph & TOP) ? 1 : 0;
        score -= (Mh & TOP) ? 1 : 0;
        Ph = ((Ph << 2) | 1u) & EVEN;   // the row above the matrix grows by one per column (global alignment)
        Mh = (Mh << 2) & EVEN;
        Pv = (Mh | ~(Xv | Ph)) & EVEN;
        Mv = Ph & Xv;
        if (j == 14) score15 = score;
    }
    Dist3 r;
    r.full = score;
    r.b15 = score15;
    r.a15 = score - ((Pv & TOP) ? 1 : 0) + ((Mv & TOP) ? 1 : 0);
    return r;
}

BDG_HD int dist3_min(uint32_t a, uint32_t b)
{
    Dist3 r = myers3(a, b);
    int d = r.full < r.a15 ? r.full : r.a15;
    return d < r.b15 ? d : r.b15;
}

// ---------------------------------------------------------------------------------------------
// S(a,b): number of (p,q) with the 6-mer of a at p equal to the 6-mer of b at q, p,q in 0..10, summed
// diagonal by diagonal (q - p = s, s = -10..10): a 6-mer match at p on diagonal s is a run of six
// matching bases starting at p.  multiplicity out: per query position p the number of matching q
// (kmer_indexer.py:53-55 `positions`), packed 4 bits per position into a uint64.
// ---------------------------------------------------------------------------------------------
BDG_HD uint32_t run6(uint32_t m)   // m: match marks; result bit 2p set <=> columns p..p+5 all match
{
    const uint32_t m2 = m & (m >> 2);
    const uint32_t m4 = m2 & (m2 >> 4);
    return m4 & (m2 >> 8);
}

BDG_HD int qgram_score(uint32_t a, uint32_t b, uint64_t* mult = nullptr)
{
    int s = 0;
    uint64_t mu = 0;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int k = 0; k <= 10; k++) {
        // diagonal +k: a[i] vs b[i+k], valid a-columns 0..15-k
        {
            const uint32_t valid = EVEN >> (2 * k);
            const uint32_t r = run6(~mism(a, b >> (2 * k)) & valid);
            s += popc(r);
            if (mult) for (int p = 0; p <= 10; p++) mu += (uint64_t)((r >> (2 * p)) & 1u) << (4 * p);
        }
        if (k == 0) continue;
        // diagonal -k: a[i] vs b[i-k], valid a-columns k..15
        {
            const uint32_t valid = EVEN << (2 * k);
            const uint32_t r = run6(~mism(a, b << (2 * k)) & valid);
            s += popc(r);
            if (mult) for (int p = 0; p <= 10; p++) mu += (uint64_t)((r >> (2 * p)) & 1u) << (4 * p);
        }
    }
    if (mult) *mult = mu;
    return s;
}

// Does the 6-mer at position p of w occur at an earlier position of w?  (Posting lists hold a string once per distinct 6-mer,
// and a query walks a bucket once per distinct 6-mer of its own.)
BDG_HD bool kmer_seen_before(uint32_t w, int p)
{
    const uint32_t k = (w >> (2 * p)) & 0xFFFu;
    bool seen = false;
    for (int e = 0; e < p; e++) seen = seen || ((w >> (2 * e)) & 0xFFFu) == k;
    return seen;
}

// The score together with the set of query positions p whose 6-mer occurs anywhere in b (bit 2p of *marks): the posting-list form
// of kmer_indexer.py:49-61 emits a (query, entry) pair from the bucket of the FIRST such position only.
BDG_HD int qgram_score_marks(uint32_t a, uint32_t b, uint32_t* marks)
{
    int s = 0;
    uint32_t any = 0;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int k = 0; k <= 10; k++) {
        {
            const uint32_t r = run6(~mism(a, b >> (2 * k)) & (EVEN >> (2 * k)));
            s += popc(r);
            any |= r;
        }
        if (k == 0) continue;
        {
            const uint32_t r = run6(~mism(a, b << (2 * k)) & (EVEN << (2 * k)));
            s += popc(r);
            any |= r;
        }
    }
    *marks = any;
    return s;
}

// Two halves of the score for the join kernel: the three middle diagonals, where nearly all of a close pair's shared 6-mers
// sit (their count alone usually reaches the threshold), and the other eighteen as a compact loop.  near + far == qgram_score.
BDG_HD int qgram_score_near(uint32_t a, uint32_t b)
{
    return popc(run6(~mism(a, b) & EVEN)) + popc(run6(~mism(a, b >> 2) & (EVEN >> 2))) + popc(run6(~mism(a, b << 2) & (EVEN << 2)));
}
BDG_HD int qgram_score_far(uint32_t a, uint32_t b)
{
    int s = 0;
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
    for (int k = 2; k <= 10; k++)
        s += popc(run6(~mism(a, b >> (2 * k)) & (EVEN >> (2 * k)))) + popc(run6(~mism(a, b << (2 * k)) & (EVEN << (2 * k))));
    return s;
}

// The same score as a compact loop (one diagonal pair per trip, nothing unrolled): the join kernel keeps its whole hot path
// inside the instruction cache, and 21 unrolled diagonals are a third of it.
BDG_HD int qgram_score_compact(uint32_t a, uint32_t b)
{
    int s = popc(run6(~mism(a, b) & EVEN));
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
    for (int k = 1; k <= 10; k++)
        s += popc(run6(~mism(a, b >> (2 * k)) & (EVEN >> (2 * k)))) + popc(run6(~mism(a, b << (2 * k)) & (EVEN << (2 * k))));
    return s;
}

BDG_HD uint32_t low_mask(int n) { return n >= 32 ? 0xFFFFFFFFu : ((1u << n) - 1u); }

// Full predicate of barcode_graph.py:233-249 for a != b: returns D when (a,b) is an edge at threshold t,
// else 0.  t <= 2 uses the case analysis, larger t the generic bit-vector pass.
BDG_HD int edge_dist(uint32_t a, uint32_t b, int t)
{
    if (t <= 0) return 0;
    int d = t <= 2 ? dist_small(a, b) : dist3_min(a, b);
    if (d > t || d == 0) return 0;
    return qgram_score(a, b) >= qgram_threshold(t) ? d : 0;
}

}  // namespace bdg
