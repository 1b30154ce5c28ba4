// Counts of the t = 2 join on the host, with the kernel's own per-pair functions (bdg_seed.cuh): per condition, every pair of
// equal-key buckets through the three-diagonal quick test with the flag table (quick_marks, seed_lut_build: the form before
// the side filter) and through the side filter with the side-aware table (join2_quick, seed_lut_build_sides).
// Built and run by tools/join_candidates_host.py.  Input: the sorted distinct barcodes as raw little-endian uint32.
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <vector>
#include <algorithm>
#include "bdg_seed.cuh"
using namespace bdg;

enum { PAIRS, CAND_OLD, CAND_NEW, NEAR_OLD, NEAR_NEW, EDGES_OLD, EDGES_NEW, NCOUNT };

int main(int argc, char** argv)
{
    if (argc < 2) { fprintf(stderr, "usage: %s barcodes.u32 [bases per block ...]\n", argv[0]); return 2; }
    FILE* f = fopen(argv[1], "rb");
    if (!f) { perror(argv[1]); return 2; }
    std::vector<uint32_t> s;
    uint32_t v;
    while (fread(&v, 4, 1, f) == 1) s.push_back(v);
    fclose(f);
    const uint32_t N = (uint32_t)s.size();
    int bases[SEED_MAX_BLOCKS] = {3, 3, 3, 3, 3}, nb = 5;
    if (argc > 2) { nb = 0; for (int i = 2; i < argc && nb < SEED_MAX_BLOCKS; i++) bases[nb++] = atoi(argv[i]); }
    SeedScheme S;
    if (!seed_scheme_build(S, bases, nb)) { fprintf(stderr, "not a usable block layout\n"); return 2; }
    std::vector<uint8_t> lut(1u << S.nflags), lut_sides(1u << (S.nflags + 2));
    seed_lut_build(S, lut.data());
    seed_lut_build_sides(S, lut_sides.data());
    std::vector<unsigned long long> T((size_t)S.nconds * NCOUNT, 0);
#pragma omp parallel for schedule(dynamic, 1)
    for (int c = 0; c < S.nconds; c++) {
        const uint32_t nk = 1u << S.ka[c].key_bits;
        auto bucket = [&](const SeedKey& k, std::vector<uint32_t>& out, std::vector<uint32_t>& st) {
            st.assign(nk + 1, 0);
            for (uint32_t x : s) st[seed_key(x, k) + 1]++;
            for (uint32_t i = 0; i < nk; i++) st[i + 1] += st[i];
            std::vector<uint32_t> pos(st.begin(), st.end() - 1);
            out.resize(N);
            for (uint32_t x : s) out[pos[seed_key(x, k)]++] = x;
        };
        std::vector<uint32_t> R, RS, C, CS;
        bucket(S.ka[c], R, RS);
        const bool self = S.cond[c].self != 0;
        if (!self) bucket(S.kb[c], C, CS);
        unsigned long long* t = &T[(size_t)c * NCOUNT];
        for (uint32_t k = 0; k < nk; k++) {
            for (uint32_t i = RS[k]; i < RS[k + 1]; i++) {
                const uint32_t x = R[i];
                const uint32_t j0 = self ? i + 1 : CS[k], j1 = self ? RS[k + 1] : CS[k + 1];
                for (uint32_t j = j0; j < j1; j++) {
                    const uint32_t y = self ? R[j] : C[j];
                    if (x == y) continue;
                    t[PAIRS]++;
                    const bool q_old = quick_pass(x, y, 2);
                    const bool q_new = self ? join2_quick<false>(x, y, y >> 2, y << 2, 1u, 0xFFFFFFFFu)
                                            : join2_quick<true>(x, y, y >> 2, y << 2, 1u, 0xFFFFFFFFu);
                    t[CAND_OLD] += q_old;
                    t[CAND_NEW] += q_new;
                    if (!q_old && !q_new) continue;
                    const uint32_t a = std::min(x, y), b = std::max(x, y);
                    if (dist_small(a, b, false, true) > 2) continue;
                    t[NEAR_OLD] += q_old;
                    t[NEAR_NEW] += q_new;
                    if (qgram_score_compact(a, b) < qgram_threshold(2)) continue;
                    const int want = 2 * c + (self || x < y ? 0 : 1);
                    t[EDGES_OLD] += q_old && lut[seed_flags(S, a, b)] == want;
                    t[EDGES_NEW] += q_new && lut_sides[seed_flags(S, a, b) | seed_side_bits(a, b) << S.nflags] == want;
                }
            }
        }
    }
    // one line per condition, then the sums over the symmetric conditions, the shifted ones and all
    unsigned long long sum[3][NCOUNT] = {};
    for (int c = 0; c < S.nconds; c++) {
        printf("cond %2d %s", c, S.cond[c].self ? "sym" : "shf");
        for (int q = 0; q < NCOUNT; q++) {
            printf(" %llu", T[(size_t)c * NCOUNT + q]);
            sum[S.cond[c].self ? 0 : 1][q] += T[(size_t)c * NCOUNT + q];
            sum[2][q] += T[(size_t)c * NCOUNT + q];
        }
        printf("\n");
    }
    const char* name[3] = {"symmetric", "shifted", "all"};
    for (int g = 0; g < 3; g++) {
        printf("total %s", name[g]);
        for (int q = 0; q < NCOUNT; q++) printf(" %llu", sum[g][q]);
        printf("\n");
    }
    printf("N %u\n", N);
    return 0;
}
