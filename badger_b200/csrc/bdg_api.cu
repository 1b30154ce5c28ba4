// bdg_api.cu -- C ABI of libbadger_b200.so (see include/badger_b200.h for the contract and the
// reference call sites each entry point replaces).  Host side only: contexts, buffers, work plans,
// launches.  All arithmetic lives in bdg_kernels.cuh / bdg_core.cuh.  There is no CPU fallback.
#include <algorithm>
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <ctime>
#include <mutex>
#include <new>
#include <string>
#include <thread>
#include <vector>

#include "../../include/badger_b200.h"
#include "bdg_kernels.cuh"
#include "bdg_join.cuh"
#include "bdg_tsv.hpp"

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <cub/device/device_select.cuh>
#include <thrust/iterator/counting_iterator.h>
#include <thrust/iterator/transform_iterator.h>

namespace {

thread_local char g_err[512] = "";
std::atomic<unsigned long long> g_launches{0};

int fail(int code, const char* fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

#define CU_TRY(expr)                                                                                   \
    do {                                                                                               \
        cudaError_t e_ = (expr);                                                                       \
        if (e_ != cudaSuccess)                                                                         \
            return fail(e_ == cudaErrorMemoryAllocation ? BDG_ERR_OOM : BDG_ERR_CUDA, "%s failed: %s", \
                        #expr, cudaGetErrorString(e_));                                                \
    } while (0)

// grow-only device buffer: the host-buffer entry points reuse their workspaces from call to call
// (cudaMalloc / cudaFree per call cost far more than the kernels at BASELINE config-2 sizes).  It owns its allocation: the
// owner makes the buffer's device current before destroying it.
struct Buf {
    void* p = nullptr;
    size_t cap = 0;
    Buf() = default;
    Buf(Buf&& o) noexcept : p(o.p), cap(o.cap) { o.p = nullptr; o.cap = 0; }
    Buf& operator=(Buf&&) = delete;
    ~Buf() { release(); }
    // at least `bytes` bytes; growing frees the old contents.  BDG_ERR_OOM / BDG_ERR_CUDA with the message set on failure.
    int ensure(size_t bytes)
    {
        if (bytes <= cap) return BDG_OK;
        release();
        const size_t want = bytes + bytes / 4 + 256;
        if (cudaError_t e = cudaMalloc(&p, want)) {
            p = nullptr;
            return fail(e == cudaErrorMemoryAllocation ? BDG_ERR_OOM : BDG_ERR_CUDA, "device allocation of %zu bytes: %s", bytes,
                        cudaGetErrorString(e));
        }
        cap = want;
        return BDG_OK;
    }

private:
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

// the work plan of one part (built by build_plan below)
struct Plan {
    std::vector<uint32_t> group_ids;
    std::vector<uint32_t> item_start;
    uint32_t chunk_cols = 256;
    uint64_t pairs = 0;
};

// The read map a dedup call leaves on the first device, named by its token, and the clustering result that may belong to it.
// Its arrays are the dedup workspaces after dedup_core, which reuses them within a call; merge and tally install theirs there.
struct ReadMap {
    Buf dd[10];                   // dedup_core's workspaces (see there); the map's arrays by name below
    Buf valid, valid_scan;        // masked dedup: the rows' valid bytes and their exclusive scan (a valid row's index among the valid rows)
    Buf centre, level;            // the last clustering on this device (cluster_on_device): centre index and level per node
    unsigned long long token = 0, serial = 0;   // token of the live read map (0: none), last token issued
    unsigned long long cl_token = 0;            // read-map token the clustering result belongs to (0: none)
    size_t rows = 0, reads = 0, distinct = 0;   // rows of the dedup call, valid rows among them, distinct barcodes (the nodes)
    bool masked = false;                        // the rows came with valid bytes

    Buf& keys() { return dd[0]; }                                      // dedup_core's input: the key of every valid read
    uint32_t* counts() const { return (uint32_t*)dd[0].p; }            // count of every distinct barcode, first-seen order
    uint32_t* order() const { return (uint32_t*)dd[1].p; }             // first-seen position -> ascending position (node)
    uint32_t* first_seen() const { return (uint32_t*)dd[2].p; }        // the distinct barcodes in first-seen order
    uint32_t* run_pos() const { return (uint32_t*)dd[4].p; }           // node -> first-seen position (dedup calls only)
    uint32_t* ascending() const { return (uint32_t*)dd[6].p; }         // the distinct barcodes ascending: the nodes
    uint32_t* read_pos() const { return (uint32_t*)dd[7].p; }          // valid read -> first-seen position (`reads` entries)

    void drop() { token = 0; cl_token = 0; }   // the workspaces are about to be reused: the live read map dies here

    // Installs a distinct set of n barcodes as the live read map and issues its token: the four arrays counts, order, first-seen,
    // ascending (as named above) hold n entries afterwards.  The sources (device arrays on this map's device) are copied in on
    // st; NULL: the array is already in place, or the caller writes it on st right after the install.
    int install(size_t n, const uint32_t* src_counts, const uint32_t* src_order, const uint32_t* src_first_seen,
                const uint32_t* src_ascending, cudaStream_t st, unsigned long long* out_token)
    {
        drop();
        CU_TRY(cudaStreamSynchronize(st));          // growing a buffer frees its old memory: queued work may still read it
        const uint32_t* src[4] = {src_counts, src_order, src_first_seen, src_ascending};
        const int slot[4] = {0, 1, 2, 6};
        for (int k = 0; k < 4; k++) {
            if (int e = dd[slot[k]].ensure(n * 4)) return e;
            if (src[k]) CU_TRY(cudaMemcpyAsync(dd[slot[k]].p, src[k], n * 4, cudaMemcpyDeviceToDevice, st));
        }
        distinct = n;
        token = ++serial;
        *out_token = token;
        return BDG_OK;
    }
};

struct DevCtx {
    int dev = -1;
    cudaStream_t stream = nullptr;
    int sms = 0;
    Buf sorted, ea, eb, ed, count, plan;   // edge construction
    // sparse passes run side by side on their own streams, so each has its own rotated keys, sorted copy, radix-sort scratch,
    // sub-tile end keys and list of tiles that survive level 1
    Buf rot_in[bdg::MAX_PASSES], rot_sorted[bdg::MAX_PASSES], sort_tmp[bdg::MAX_PASSES], tile_bnd[bdg::MAX_PASSES], tile_list[bdg::MAX_PASSES];
    cudaStream_t aux[bdg::MAX_PASSES] = {nullptr, nullptr, nullptr};   // aux[p]: stream of pass p (pass 0 stays on the caller's stream)
    cudaEvent_t ev_start = nullptr, ev_done[bdg::MAX_PASSES] = {nullptr, nullptr, nullptr};
    unsigned long long host_stats[bdg::MAX_PASSES][2] = {};   // interval tests done / tiles listed per pass of the last launch
    unsigned long long generation = 0;                        // bumped by every host-buffer edge build on this device
    ReadMap map;                                              // the read map of the last dedup call (first device)
    Buf io;                                                   // one call's uploads, outputs and per-read scratch, carved by stage() (see there)
    Buf sort_flag;                                            // whitelist check: index of the first entry not above its predecessor
    Buf cl_centres, cl_min, cl_max, cl_flags;                 // clustering: centres, claim min / max, flags + count (result: map.centre / map.level)
    // centre selection (centres_above, centres_rest) and pack16_sorted, which runs in the same buffers
    Buf sel;                                                  // positions above the cutoff | pack16_sorted: the valid records' ranks
    Buf sel_keys;                                             // their sort keys | the ranks sorted
    Buf sel_sorted;                                           // the sort keys sorted | the distinct ranks (pack16_sorted's result)
    Buf sel_scalars;                                          // count sum and selection size | the number of ranks kept
    Buf sel_tmp;                                              // cub scratch of both
    Buf sel_pos, head_ranks, head_counts, head_hits;          // centre selection: positions in count order, the head, its counts and hits
    Buf mask_tmp;                                             // masked dedup: cub scratch of the scan of the valid bytes
    Buf centre_val;                                           // per-read gathers: centre value + has byte per distinct barcode
    Buf counters;                                             // per-read gathers: rows with a centre (assign_reads32) | assigned, missing (assign_lookup32)
    struct {                                                  // merge of the parts' dedup results (bdg_dev_dedup_merge), see there
        Buf starts, offs, key, idx, sorted_key, sorted_idx, cnt, first, head, scan, runs, tmp;
    } mg;
    Buf gather_a, gather_b;                                   // node indices of the edge ends: this device's own, and (first device) those of ALL devices, gathered for cluster()
    Buf top16;                                                // first node of every high half of the barcode (the node of an edge end is searched in that run)
    struct NearSide { Buf key, pay, key_sorted, pay_sorted; };
    NearSide nn_q, nn_t;                                      // sparse nearest: rotated keys + payload (in / sorted) of the queries and the targets
    Buf nn_tmp;                                               // sparse nearest: radix-sort scratch
    // join form of the t = 2 and t = 3 edge construction (bdg_join.cuh): barcodes in the key order of every condition's row side /
    // column side, first column of every key, bucket sizes and every barcode's place in its bucket, scan scratch, units per slab
    // and their prefix sums (one set per stream: the conditions of a block set run back to back on one stream); the t = 2
    // hand-over table and the work-estimate histograms
    Buf jn_rows[2], jn_cols[2], jn_tab[2], jn_tabc[2], jn_hist[2], jn_cub[2], jn_counts[2], jn_offs[2], jn_rank[2], jn_lut, jn_weigh;
    int scheme_serial = 0;                                    // which t = 2 scheme sits in this device's constant memory (0: none)
    Buf jn3_scheme;                                           // t = 3 join: device copy of the seed table (bdg_seed3.cuh)
    int scheme3_serial = 0;
    cudaEvent_t ev_snap[bdg::JOIN_MAX_SNAPS] = {};            // bdg_edges_build_into: "the edges up to snapshot q are appended"
    cudaEvent_t ev_pre[2] = {nullptr, nullptr}, ev_join[2] = {nullptr, nullptr};   // streaming form: scratch set k is bucketed / its join has finished
    unsigned long long* snap_host = nullptr;                  // mapped page-locked: the edge count at every snapshot
    unsigned long long* snap_dev = nullptr;
    cudaEvent_t ev_caller = nullptr;                          // bdg_dev_* correction-step calls: orders this device's stream against the caller's
};
// Never deleted: the buffers are freed by bdg_shutdown, not by static destructors at process exit.
std::vector<DevCtx>& g_ctx = *new std::vector<DevCtx>;

int owner_of_tile(uint64_t I, int P)
{
    const uint64_t m = I % (2ull * P);
    return (int)(m < (uint64_t)P ? m : 2ull * P - 1 - m);
}

int grid_for(const void* kernel, int* out, int threads = bdg::NT)
{
    int dev = 0, sms = 0, occ = 0;
    CU_TRY(cudaGetDevice(&dev));
    CU_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    CU_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, threads, 0));
    if (occ < 1) occ = 1;
    *out = sms * occ;
    return BDG_OK;
}

// ---- the work plan of one part: owned row groups (256 rows, one warp each), column chunks per group ----
// Ownership is dealt in tiles of BDG_ROW_TILE rows (8 groups), boustrophedon over the parts.
void build_plan(size_t N, int part, int nparts, int workers, Plan& p, uint64_t col_quantum = bdg::SB_MAX)
{
    const uint64_t tiles = (N + bdg::ROW_TILE - 1) / bdg::ROW_TILE;
    const uint64_t groups = (N + bdg::GROUP - 1) / bdg::GROUP;
    constexpr uint64_t GPT = bdg::ROW_TILE / bdg::GROUP;
    p.group_ids.clear();
    p.pairs = 0;
    for (uint64_t I = 0; I < tiles; I++) {
        if (owner_of_tile(I, nparts) != part) continue;
        const uint64_t r0 = I * bdg::ROW_TILE, r1 = std::min<uint64_t>(N, r0 + bdg::ROW_TILE);
        const uint64_t n = r1 - r0;                       // rows i in [r0,r1): N-1-i partners each
        p.pairs += n * (N - 1) - (r0 + r1 - 1) * n / 2;
        for (uint64_t g = I * GPT; g < std::min(groups, (I + 1) * GPT); g++) p.group_ids.push_back((uint32_t)g);
    }
    // aim at >= 16 work items per resident warp so that the dynamic scheduler can level the load
    double per_worker = 16.0;
    if (const char* e = getenv("BDG_EDGE_ITEMS")) per_worker = std::max(1.0, atof(e));
    const double want_items = per_worker * std::max(workers, 1);
    const double cols = ((double)p.pairs / bdg::GROUP) / want_items;
    uint64_t cc = (uint64_t)cols / col_quantum * col_quantum;
    cc = std::min<uint64_t>(std::max<uint64_t>(cc, std::max<uint64_t>(col_quantum, 4 * bdg::SB_MAX)), 1u << 17);
    p.chunk_cols = (uint32_t)cc;
    p.item_start.assign(p.group_ids.size() + 1, 0);
    uint64_t acc = 0;
    for (size_t k = 0; k < p.group_ids.size(); k++) {
        p.item_start[k] = (uint32_t)acc;
        const uint64_t ncols = N - (uint64_t)p.group_ids[k] * bdg::GROUP;
        acc += (ncols + cc - 1) / cc;
    }
    p.item_start[p.group_ids.size()] = (uint32_t)acc;
}

constexpr size_t PLAN_HDR = 128;  // per launch: [work cursor u64 | tile-list count u64 | 8 x u64 statistics | pad]
constexpr size_t HDR_LIST = 8, HDR_STATS = 16;
int g_edge_mode = -1;             // -1: BDG_EDGE_MODE or default (by threshold and size); 0 dense; 1 sparse; 2 join
constexpr size_t JOIN3_MIN_N = 90000;   // t = 3: join from this many distinct barcodes upwards (measured crossover, DESIGN.md 3.8)

// 0 dense, 1 sparse, 2 join.  The join form exists for t = 2 and t = 3 and pays off once the key buckets fill (DESIGN.md 3);
// below that t = 2 runs sparse and t = 3, which has no sparse form, dense.
int edge_mode_for(int t, size_t N)
{
    int m = g_edge_mode;
    if (m < 0) {
        const char* e = getenv("BDG_EDGE_MODE");
        if (e && !strcmp(e, "dense")) m = 0;
        else if (e && !strcmp(e, "sparse")) m = 1;
        else if (e && !strcmp(e, "join")) m = 2;
        else if (t == 2 || t == 3) {
            size_t min_n = t == 2 ? 150000 : JOIN3_MIN_N;
            if (const char* j = getenv(t == 2 ? "BDG_JOIN_MIN_N" : "BDG_JOIN3_MIN_N")) min_n = (size_t)std::max(0ll, atoll(j));
            m = N >= min_n ? 2 : t == 2 ? 1 : 0;
        } else m = t == 1 ? 1 : 0;
    }
    if (m == 2 && (t < 2 || t > 3 || N >= (1ull << 28))) m = t == 3 ? 0 : 1;
    if (m == 1 && t != 1 && t != 2) m = 0;
    return m;
}

// ---- the seed schemes of the join form: built once on the host (bdg_seed.cuh, bdg_seed3.cuh), copied to every device that uses them ----
bdg::SeedScheme g_scheme;
std::vector<uint8_t> g_scheme_lut;
bdg::Seed3Scheme g_scheme3;
int g_scheme_serial = 0, g_scheme3_serial = 0;

std::mutex g_scheme_mutex;        // the devices of one build call arrive on their own host threads

template <int T>
const auto& join_scheme()
{
    if constexpr (T == 2) return g_scheme; else return g_scheme3;
}

// The block layout of the threshold-T table is BDG_JOIN_BLOCKS / BDG_JOIN3_BLOCKS (e.g. "4,4,4,3" / "3,3,3,2,2,2": development
// aids), else five blocks of 3 bases at t = 2 and 3,2,2,2,2,2,2 at t = 3.
template <int T>
int scheme_ready()
{
    std::lock_guard<std::mutex> lock(g_scheme_mutex);
    int& serial = T == 2 ? g_scheme_serial : g_scheme3_serial;
    if (serial) return BDG_OK;
    const int max_blocks = T == 2 ? bdg::SEED_MAX_BLOCKS : bdg::SEED3_MAX_BLOCKS;
    int bases[bdg::SEED3_MAX_BLOCKS] = {3, 3, 3, 3, 3, 3, 3};
    int nb = T == 2 ? 5 : 7;
    if (T == 3) std::fill(bases + 1, bases + nb, 2);
    if (const char* e = getenv(T == 2 ? "BDG_JOIN_BLOCKS" : "BDG_JOIN3_BLOCKS")) {
        nb = 0;
        for (const char* p = e; *p && nb < max_blocks;) {
            bases[nb++] = atoi(p);
            while (*p && *p != ',') p++;
            if (*p == ',') p++;
        }
    }
    if constexpr (T == 2) {
        if (!bdg::seed_scheme_build(g_scheme, bases, nb)) return fail(BDG_ERR_ARG, "BDG_JOIN_BLOCKS is not a usable block layout (3..6 blocks, 15 bases in all)");
        g_scheme_lut.assign((size_t)1 << (g_scheme.nflags + 2), 0);          // block-match flags and the two side bits
        bdg::seed_lut_build_sides(g_scheme, g_scheme_lut.data());
    } else {
        if (!bdg::seed3_scheme_build(g_scheme3, bases, nb)) return fail(BDG_ERR_ARG, "BDG_JOIN3_BLOCKS is not a usable block layout (4..7 blocks of >= 2 bases, 15 bases in all)");
    }
    serial = 1;
    return BDG_OK;
}

template <int T_, int P_>
void launch_scan(int blocks, cudaStream_t st, const bdg::EdgeWork& w, const uint2* bnd, uint32_t NS, const bdg::TileList& l)
{
    bdg::sparse_scan_kernel<T_, P_, false><<<blocks, 256, 0, st>>>(w.sorted, w.N, w.group_ids, w.K, bnd, NS, l);
}
template <int T_, int P_>
void launch_tiles(int blocks, cudaStream_t st, const bdg::EdgeWork& w, const bdg::EdgeOut& o, const bdg::TileList& l)
{
    bdg::sparse_tile_kernel<T_, P_, false><<<blocks, bdg::ENT, 0, st>>>(w, o, l);
}
template <int T_, int P_>
void launch_scan_bip(int blocks, cudaStream_t st, const bdg::EdgeWork& w, const uint2* bnd, uint32_t NS, const bdg::TileList& l)
{
    bdg::sparse_scan_kernel<T_, P_, true><<<blocks, 256, 0, st>>>(w.sorted, w.N, nullptr, w.K, bnd, NS, l);
}
template <int T_, int P_>
void launch_tiles_bip(int blocks, cudaStream_t st, const bdg::EdgeWork& w, const bdg::EdgeOut& o, const bdg::TileList& l)
{
    bdg::sparse_tile_kernel<T_, P_, true><<<blocks, bdg::ENT, 0, st>>>(w, o, l);
}
#define BDG_PASS_DISPATCH(FN, ...)                                                    \
    do {                                                                              \
        if (t == 1) { if (p == 0) FN<1, 0>(__VA_ARGS__); else FN<1, 1>(__VA_ARGS__); } \
        else if (p == 0) FN<2, 0>(__VA_ARGS__);                                       \
        else if (p == 1) FN<2, 1>(__VA_ARGS__);                                       \
        else FN<2, 2>(__VA_ARGS__);                                                   \
    } while (0)

double now_ms()
{
    timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return ts.tv_sec * 1e3 + ts.tv_nsec * 1e-6;
}

// Join form (t = 2 and t = 3), bdg_join.cuh.  The seed conditions are laid on a line by weight (their estimated work, see below)
// and the line is cut into nparts equal pieces: a part sorts and joins only the conditions its piece touches, a condition on a
// cut is shared by row range (cut at a bucket boundary).  Per condition: counting sort by the key (rows once per block set,
// columns for the shifted conditions; its prefix sums are colstart) -> units per slab -> prefix sums -> one persistent join
// launch.  The conditions of a block set follow one another and share the row order.  Consecutive block sets alternate between
// the caller's stream and an auxiliary one, so that one condition's sorts and the tail of its join overlap the neighbour's join.
// Host buffers the finished edges are copied into WHILE later conditions still run (bdg_edges_build_into): the conditions
// then run on one stream, a snapshot of the edge count follows every condition (t = 2) or the last condition of every block
// set (t = 3, whose 475 conditions are short), and the ranges between two snapshots - final, because their launches have
// ended - leave on the copy stream.
struct JoinStream {
    uint32_t* h_a;
    uint32_t* h_b;
    uint8_t* h_d;
    size_t h_cap;
};

template <int T>
int launch_edges_join(const uint32_t* d_sorted, size_t N, int part, int nparts, uint32_t* d_a, uint32_t* d_b, uint8_t* d_d, size_t cap,
                      unsigned long long* d_count, cudaStream_t caller, DevCtx* ws, const JoinStream* js)
{
    if (int rc = scheme_ready<T>()) return rc;
    const auto& S = join_scheme<T>();
    if constexpr (T == 2) {                                 // the table to constant memory, the hand-over table beside it
        if (ws->scheme_serial != g_scheme_serial) {
            if (int e = ws->jn_lut.ensure(g_scheme_lut.size())) return e;
            CU_TRY(cudaMemcpyToSymbolAsync(bdg::c_scheme, &g_scheme, sizeof(g_scheme), 0, cudaMemcpyHostToDevice, caller));
            CU_TRY(cudaMemcpyAsync(ws->jn_lut.p, g_scheme_lut.data(), g_scheme_lut.size(), cudaMemcpyHostToDevice, caller));
            CU_TRY(cudaStreamSynchronize(caller));          // the host copies above are read asynchronously
            ws->scheme_serial = g_scheme_serial;
        }
    } else {                                                // too large for constant memory: a device copy
        if (ws->scheme3_serial != g_scheme3_serial) {
            if (int e = ws->jn3_scheme.ensure(sizeof(g_scheme3))) return e;
            CU_TRY(cudaMemcpyAsync(ws->jn3_scheme.p, &g_scheme3, sizeof(g_scheme3), cudaMemcpyHostToDevice, caller));
            CU_TRY(cudaStreamSynchronize(caller));          // the host copy above is read asynchronously
            ws->scheme3_serial = g_scheme3_serial;
        }
    }
    // rows per sub-slab: 8 when the key buckets are short (fewer rows then span fewer foreign buckets), else 32
    int rs = (N >> S.ka[0].key_bits) < 48 ? 8 : 32;
    if (const char* e = getenv("BDG_JOIN_RS")) rs = atoi(e) == 8 ? 8 : 32;
    const uint32_t n_slabs = (uint32_t)((N + bdg::JROWS - 1) / bdg::JROWS);
    const bool trace = getenv("BDG_TRACE") != nullptr;
    // Weights of the conditions for the deal to the parts: one part takes everything; several parts estimate every condition's
    // pairs from bucket sizes over a sample (identical integer arithmetic on every part) and add the bucketing of its sides.
    std::vector<long long> weight(S.nconds, 1);
    const double t_weigh = trace ? (cudaStreamSynchronize(caller), now_ms()) : 0.0;
    if (nparts > 1 || trace) {                              // (traced runs print the estimate beside the measured time of every condition)
        const uint32_t stride = (uint32_t)std::max<size_t>(1, (N + (1u << 17) - 1) >> 17);
        const uint32_t m = (uint32_t)((N + stride - 1) / stride);
        const int hb = (int)std::min<uint32_t>((m + 255) / 256, (uint32_t)ws->sms * 8);
        unsigned long long* d_pairs = nullptr;
        if constexpr (T == 2) {                             // all tables in one pass
            uint32_t maxtab = 4;
            for (int c = 0; c < S.nconds; c++) maxtab = std::max(maxtab, 1u << S.ka[c].key_bits);
            bdg::WeighSlots slots{};
            for (int c = 0; c < S.nconds; c++) {
                slots.row[c] = S.cond[c].row_sort == c ? (uint8_t)slots.n++ : slots.row[S.cond[c].row_sort];
                slots.col[c] = S.cond[c].self ? slots.row[c] : (uint8_t)slots.n++;
            }
            const size_t hist_bytes = (size_t)slots.n * maxtab * 4;
            if (int e = ws->jn_weigh.ensure(hist_bytes + 8 * bdg::SEED_MAX_CONDS)) return e;
            uint32_t* d_hist = (uint32_t*)ws->jn_weigh.p;
            d_pairs = (unsigned long long*)((char*)ws->jn_weigh.p + hist_bytes);
            CU_TRY(cudaMemsetAsync(ws->jn_weigh.p, 0, hist_bytes + 8 * bdg::SEED_MAX_CONDS, caller));
            bdg::join_weigh_hist_kernel<<<hb, 256, 0, caller>>>(d_sorted, (uint32_t)N, stride, S.nconds, maxtab, slots, d_hist);
            bdg::join_weigh_sum_kernel<<<dim3((maxtab / 4 + 1023) / 1024, S.nconds), 256, 0, caller>>>(d_hist, maxtab, slots, d_pairs);
            g_launches += 2;
        } else {                                            // block set by block set: one row table and the set's column tables at a time
            int max_set = 1, max_bits = 0;
            for (int k = 0; k < S.nsets; k++) max_set = std::max(max_set, (int)(S.set_first[k + 1] - S.set_first[k]));
            for (int c = 0; c < S.nconds; c++) max_bits = std::max(max_bits, (int)S.ka[c].key_bits);
            const uint32_t tab = 1u << max_bits;
            const size_t hist_bytes = (size_t)max_set * tab * 4;
            if (int e = ws->jn_weigh.ensure(hist_bytes + 8 * (size_t)bdg::SEED3_MAX_CONDS)) return e;
            uint32_t* d_hist = (uint32_t*)ws->jn_weigh.p;
            d_pairs = (unsigned long long*)((char*)ws->jn_weigh.p + hist_bytes);
            CU_TRY(cudaMemsetAsync(d_pairs, 0, 8 * (size_t)S.nconds, caller));
            for (int k = 0; k < S.nsets; k++) {
                const int c0 = S.set_first[k], c1 = S.set_first[k + 1];
                CU_TRY(cudaMemsetAsync(d_hist, 0, (size_t)(c1 - c0) * tab * 4, caller));
                bdg::join3_weigh_hist_kernel<<<hb, 256, 0, caller>>>(d_sorted, (uint32_t)N, stride, (const bdg::Seed3Scheme*)ws->jn3_scheme.p, c0, c1, tab, d_hist);
                bdg::join3_weigh_sum_kernel<<<dim3((tab + 1023) / 1024, c1 - c0), 256, 0, caller>>>(d_hist, tab, c0, d_pairs);
                g_launches += 2;
            }
        }
        std::vector<unsigned long long> pairs(S.nconds), cost(S.nconds);
        CU_TRY(cudaMemcpyAsync(pairs.data(), d_pairs, 8 * (size_t)S.nconds, cudaMemcpyDeviceToHost, caller));
        CU_TRY(cudaStreamSynchronize(caller));
        // Cost model fitted to the per-condition times of a traced t = 2 C4 run (BDG_TRACE; 25 conditions, rms error 8 %), and
        // reused at t = 3 without refitting:
        //   time ~ pairs x (1.45 for a symmetric condition, 1 for a shifted one) + 2.4 x N.
        // A symmetric condition's pairs are counted once (n (n - 1) / 2) and hold most of the really close pairs of barcode data -
        // the ones that cost an exact distance, a hand-over check and a score sit on diagonal 0; the N term is the bucketing and
        // the per-slab bookkeeping.  Scaled to <= 4096 so that the cut arithmetic stays small.
        unsigned long long top = 1;
        for (int c = 0; c < S.nconds; c++) {
            cost[c] = pairs[c] * stride * stride * (S.cond[c].self ? 29 : 20) + 48ull * N;
            top = std::max(top, cost[c]);
        }
        for (int c = 0; c < S.nconds; c++) weight[c] = (long long)std::max<unsigned long long>(1, cost[c] * 4096 / top);
        if (trace) {
            fprintf(stderr, "[bdg] join work estimate: %.3f ms\n", now_ms() - t_weigh);
            fprintf(stderr, "[bdg] join weights (part %d of %d):", part, nparts);
            for (int c = 0; c < S.nconds; c++) fprintf(stderr, " %lld", weight[c]);
            fprintf(stderr, "\n[bdg] join estimated pairs:");
            for (int c = 0; c < S.nconds; c++) fprintf(stderr, " %llu", pairs[c] * stride * stride);
            fprintf(stderr, "\n");
        }
    }
    // Order of the conditions along the line: block set by block set (a set shares its row order), the sets taken alternately
    // from the front and from the back of the table.  A pair that meets several conditions is emitted by the first one in TABLE
    // order, so the early sets own most of the edges; alternating spreads the edges (their scores, stores and PCIe bytes) over
    // the parts.  This part keeps the conditions its piece of the line touches, with their row ranges.
    struct Piece { int c, set; long long lo, hi, c_lo, c_hi; };
    std::vector<Piece> mine;
    {
        long long W = 0, start = 0;
        for (int c = 0; c < S.nconds; c++) W += weight[c];
        const long long piece_lo = (long long)part * W, piece_hi = (long long)(part + 1) * W;   // cond c covers [start_c * nparts, (start_c + w_c) * nparts)
        for (int i = 0, lo = 0, hi = S.nsets - 1; lo <= hi; i++) {
            const int set = (i & 1) ? hi-- : lo++;
            for (int c = S.set_first[set]; c < S.set_first[set + 1]; c++) {
                const long long c_lo = start * nparts, c_hi = (start + weight[c]) * nparts;
                start += weight[c];
                const long long p_lo = std::max(c_lo, piece_lo), p_hi = std::min(c_hi, piece_hi);
                if (p_lo < p_hi) mine.push_back({c, set, p_lo, p_hi, c_lo, c_hi});
            }
        }
    }
    const size_t plan_bytes = PLAN_HDR * bdg::MAX_PASSES + 8 * (size_t)S.nconds;
    if (int e = ws->plan.ensure(plan_bytes)) return e;
    char* d_plan = (char*)ws->plan.p;
    CU_TRY(cudaMemsetAsync(d_plan, 0, plan_bytes, caller));
    for (int p = 0; p < bdg::MAX_PASSES; p++) ws->host_stats[p][0] = ws->host_stats[p][1] = 0;
    unsigned long long* d_cursors = (unsigned long long*)(d_plan + PLAN_HDR * bdg::MAX_PASSES);
    int max_bits = 0;
    for (int c = 0; c < S.nconds; c++) max_bits = std::max(max_bits, (int)S.ka[c].key_bits);
    const size_t max_keys = (size_t)1 << max_bits;
    size_t tmp_a = 0, tmp_b = 0;
    CU_TRY(cub::DeviceScan::ExclusiveSum(nullptr, tmp_a, (const uint32_t*)nullptr, (uint32_t*)nullptr, (int)(max_keys + 1), caller));
    CU_TRY(cub::DeviceScan::ExclusiveSum(nullptr, tmp_b, (const uint32_t*)nullptr, (uint32_t*)nullptr, (int)(n_slabs + 1), caller));
    const size_t tmp_bytes = std::max(tmp_a, tmp_b);
    for (int k = 0; k < 2; k++) {                           // one scratch set per stream
        if (int e = ws->jn_hist[k].ensure((max_keys + 1) * 4)) return e;
        if (int e = ws->jn_tab[k].ensure((max_keys + 1) * 4)) return e;
        if (int e = ws->jn_tabc[k].ensure((max_keys + 1) * 4)) return e;
        if (int e = ws->jn_rows[k].ensure(N * 4)) return e;
        if (int e = ws->jn_cols[k].ensure(N * 4)) return e;
        if (int e = ws->jn_rank[k].ensure(N * 4)) return e;
        if (int e = ws->jn_cub[k].ensure(tmp_bytes)) return e;
        if (int e = ws->jn_counts[k].ensure(((size_t)n_slabs + 1) * 4)) return e;
        if (int e = ws->jn_offs[k].ensure(((size_t)n_slabs + 1) * 4)) return e;
    }
    // t = 2: the shifted conditions have a kernel of their own (the one-sided test is compiled in; at t = 3 it is the same kernel);
    // both are built for the same residency, so one grid serves both
    const auto kern = rs == 8 ? bdg::join_kernel<T, 8> : bdg::join_kernel<T, 32>;
    const auto kern_shf = rs == 8 ? bdg::join_kernel<T, 8, T == 2> : bdg::join_kernel<T, 32, T == 2>;
    int grid = 0;
    if (int rc = grid_for((const void*)kern, &grid, bdg::ENT)) return rc;
    if (const char* e = getenv("BDG_JOIN_CTAS")) grid = std::min(grid, ws->sms * std::max(1, atoi(e)));   // CTAs per SM of a join launch
    const int gb = (int)std::min<size_t>((N + 255) / 256, (size_t)ws->sms * 8);
    const int bb = (int)std::min<size_t>(((size_t)n_slabs + 256) / 256, (size_t)ws->sms * 8);
    // Two ways to keep the bucketing of one condition out of the way of the joins.  The resident form forks: its two streams
    // carry whole conditions (bucketing + join) and overlap each other.  The streaming form (js) must be able to say "edges
    // [0, n) are complete" after every snapshot, so its joins stay on ONE stream in order, and only the bucketing of the next
    // condition runs ahead on a second stream, into the other scratch set.
    const bool fork = !js && !getenv("BDG_EDGE_SERIAL");
    const bool ahead = js && !getenv("BDG_EDGE_SERIAL");
    if (fork || ahead) CU_TRY(cudaEventRecord(ws->ev_start, caller));
    bool set_joined[2] = {false, false};                     // ahead: a join on scratch set k is in flight / done (ev_join[k] recorded)
    bool aux_used = false;
    int n_snaps = 0;
    if (js && !ws->snap_host) {
        CU_TRY(cudaHostAlloc((void**)&ws->snap_host, sizeof(unsigned long long) * bdg::JOIN_MAX_SNAPS, cudaHostAllocMapped));
        CU_TRY(cudaHostGetDevicePointer((void**)&ws->snap_dev, ws->snap_host, 0));
        for (int q = 0; q < bdg::JOIN_MAX_SNAPS; q++) CU_TRY(cudaEventCreateWithFlags(&ws->ev_snap[q], cudaEventDisableTiming));
        for (int q = 0; q < 2; q++) { CU_TRY(cudaEventCreateWithFlags(&ws->ev_pre[q], cudaEventDisableTiming)); CU_TRY(cudaEventCreateWithFlags(&ws->ev_join[q], cudaEventDisableTiming)); }
    }
    bdg::EdgeOut o{d_a, d_b, d_d, d_count, (unsigned long long)cap};
    int cur_set = -1, k = 1;                                 // k: scratch set / stream of the current condition
    int row_set[2] = {-1, -1};                               // block set whose row order the scratch set holds
    double t_prev = 0;
    if (trace) { cudaStreamSynchronize(caller); t_prev = now_ms(); }
    for (size_t oi = 0; oi < mine.size(); oi++) {
        const int c = mine[oi].c, set = mine[oi].set;
        // The whole job alternates its two streams block set by block set (a set sorts its rows once).  A part of several has few
        // conditions, often of one set: it alternates condition by condition, so that the bucketing of one condition runs beside
        // the join of the other, and sorts the rows again when the stream's row order is of another set.
        if (nparts > 1 || ahead || set != cur_set) k ^= 1;
        cur_set = set;
        const bool new_set = row_set[k] != set;
        row_set[k] = set;
        cudaStream_t st = (fork && k == 1) ? ws->aux[1] : caller;           // the join's stream
        cudaStream_t sp = ahead ? ws->aux[1] : st;                           // the bucketing's stream
        if (fork && k == 1 && !aux_used) { CU_TRY(cudaStreamWaitEvent(st, ws->ev_start, 0)); aux_used = true; }
        if (ahead) {
            if (!aux_used) { CU_TRY(cudaStreamWaitEvent(sp, ws->ev_start, 0)); aux_used = true; }
            if (set_joined[k]) CU_TRY(cudaStreamWaitEvent(sp, ws->ev_join[k], 0));      // the last join that read this scratch set
        }
        // counting sort of the barcodes by one side's key: bucket sizes -> first position of every key (kept: colstart) -> scatter
        auto bucket_side = [&](const bdg::SeedKey& key, Buf& dst, Buf& table) -> int {
            const size_t nkeys = (size_t)1 << key.key_bits;
            uint32_t* hist = (uint32_t*)ws->jn_hist[k].p;
            uint32_t* rank = (uint32_t*)ws->jn_rank[k].p;
            size_t bytes = ws->jn_cub[k].cap;
            CU_TRY(cudaMemsetAsync(hist, 0, (nkeys + 1) * 4, sp));
            bdg::join_hist_rank_kernel<<<gb, 256, 0, sp>>>(d_sorted, (uint32_t)N, key, hist, rank);
            CU_TRY(cub::DeviceScan::ExclusiveSum(ws->jn_cub[k].p, bytes, (const uint32_t*)hist, (uint32_t*)table.p, (int)(nkeys + 1), sp));
            bdg::join_scatter_rank_kernel<<<gb, 256, 0, sp>>>(d_sorted, (uint32_t)N, key, (const uint32_t*)table.p, rank, (uint32_t*)dst.p);
            g_launches += 2;
            return BDG_OK;
        };
        if (new_set) { if (int e = bucket_side(S.ka[S.set_first[set]], ws->jn_rows[k], ws->jn_tab[k])) return e; }      // the stream's row order: this block set
        bdg::JoinArgsT<T> A{};
        A.rows = (const uint32_t*)ws->jn_rows[k].p;
        A.rowstart = (const uint32_t*)ws->jn_tab[k].p;
        A.nkeys = 1u << S.ka[c].key_bits;
        if (S.cond[c].self) {
            A.cols = A.rows;
            A.colstart = (const uint32_t*)ws->jn_tab[k].p;
        } else {
            if (int e = bucket_side(S.kb[c], ws->jn_cols[k], ws->jn_tabc[k])) return e;
            A.cols = (const uint32_t*)ws->jn_cols[k].p;
            A.colstart = (const uint32_t*)ws->jn_tabc[k].p;
        }
        A.offs = (const uint32_t*)ws->jn_offs[k].p;
        A.cursor = d_cursors + c;
        A.stats = (unsigned long long*)(d_plan + HDR_STATS);
        A.N = (uint32_t)N;
        A.n_slabs = n_slabs;
        A.cond = c;
        A.self = S.cond[c].self;
        A.f0 = (uint32_t)(mine[oi].lo - mine[oi].c_lo); A.f1 = (uint32_t)(mine[oi].hi - mine[oi].c_lo); A.fden = (uint32_t)(mine[oi].c_hi - mine[oi].c_lo);
        A.T = bdg::qgram_threshold(T);
        A.one = 1u;
        A.mone = 0xFFFFFFFFu;
        if constexpr (T == 2) {
            A.lut = (const uint8_t*)ws->jn_lut.p;
        } else {
            A.ka = S.ka[c];
            A.kb = S.kb[c];
            A.scheme = (const bdg::Seed3Scheme*)ws->jn3_scheme.p;
        }
        bdg::join_band_kernel<T><<<bb, 256, 0, sp>>>(A, (uint32_t*)ws->jn_counts[k].p);
        size_t bytes = ws->jn_cub[k].cap;
        CU_TRY(cub::DeviceScan::ExclusiveSum(ws->jn_cub[k].p, bytes, (const uint32_t*)ws->jn_counts[k].p, (uint32_t*)ws->jn_offs[k].p, (int)(n_slabs + 1), sp));
        if (ahead) {
            CU_TRY(cudaEventRecord(ws->ev_pre[k], sp));
            CU_TRY(cudaStreamWaitEvent(st, ws->ev_pre[k], 0));
        }
        (S.cond[c].self ? kern : kern_shf)<<<grid, bdg::ENT, 0, st>>>(A, o);
        g_launches += 3;
        CU_TRY(cudaGetLastError());
        if (ahead) { CU_TRY(cudaEventRecord(ws->ev_join[k], st)); set_joined[k] = true; }
        if (trace) {                                        // development aid: per-condition wall time (serialises the streams)
            CU_TRY(cudaStreamSynchronize(st));
            const double now = now_ms();
            fprintf(stderr, "[bdg] join cond %3d (set %2d, %s, rows %u/%u..%u/%u, weight %lld): %.3f ms\n", c, set, S.cond[c].self ? "sym" : "shf",
                    A.f0, A.fden, A.f1, A.fden, weight[c], now - t_prev);
            t_prev = now;
        }
        if (js && (T == 2 || oi + 1 == mine.size() || mine[oi + 1].set != set)) {
            bdg::join_snapshot_kernel<<<1, 1, 0, st>>>(d_count, ws->snap_dev + n_snaps);
            g_launches++;
            CU_TRY(cudaEventRecord(ws->ev_snap[n_snaps], st));
            n_snaps++;
        }
    }
    if (aux_used) {
        CU_TRY(cudaEventRecord(ws->ev_done[1], ws->aux[1]));
        CU_TRY(cudaStreamWaitEvent(caller, ws->ev_done[1], 0));
    }
    if (trace) { cudaStreamSynchronize(caller); fprintf(stderr, "[bdg] join part %d of %d: %.3f ms from entry to the last condition\n", part, nparts, now_ms() - t_weigh); }
    if (js) {                                               // everything is enqueued: follow the snapshots and copy what they have finished
        cudaStream_t cp = ws->aux[2];
        size_t done = 0;
        for (int q = 0; q < n_snaps; q++) {
            CU_TRY(cudaEventSynchronize(ws->ev_snap[q]));
            const size_t upto = (size_t)std::min<unsigned long long>(ws->snap_host[q], js->h_cap);
            if (upto > done) {
                CU_TRY(cudaMemcpyAsync(js->h_a + done, d_a + done, (upto - done) * 4, cudaMemcpyDeviceToHost, cp));
                CU_TRY(cudaMemcpyAsync(js->h_b + done, d_b + done, (upto - done) * 4, cudaMemcpyDeviceToHost, cp));
                CU_TRY(cudaMemcpyAsync(js->h_d + done, d_d + done, upto - done, cudaMemcpyDeviceToHost, cp));
                done = upto;
            }
        }
        CU_TRY(cudaStreamSynchronize(cp));
    }
    return BDG_OK;
}

// Launch the edge construction of one part on the current device / stream.  d_count is zeroed on the stream.
// ws: the device's grow-only workspaces (plan, rotated keys, sort scratch); one in-flight call per device.
int launch_edges(const uint32_t* d_sorted, size_t N, int t, int part, int nparts, uint32_t* d_a, uint32_t* d_b,
                 uint8_t* d_d, size_t cap, unsigned long long* d_count, cudaStream_t st, DevCtx* ws, const JoinStream* js = nullptr)
{
    if (nparts < 1 || part < 0 || part >= nparts) return fail(BDG_ERR_ARG, "part %d of %d is not a valid part", part, nparts);
    if (N > 0xFFFFFFFFull) return fail(BDG_ERR_ARG, "N = %zu exceeds the 2^32 distinct 16-mers", N);
    if (!ws) return fail(BDG_ERR_NODEVICE, "bdg_init has not claimed the current CUDA device");
    CU_TRY(cudaMemsetAsync(d_count, 0, sizeof(unsigned long long), st));
    if (t <= 0 || N < 2) return BDG_OK;   // D >= 1 for distinct barcodes: no edges (barcode_graph.py:245)
    const int mode = edge_mode_for(t, N);
    if (mode == 2) return t == 3 ? launch_edges_join<3>(d_sorted, N, part, nparts, d_a, d_b, d_d, cap, d_count, st, ws, js)
                                 : launch_edges_join<2>(d_sorted, N, part, nparts, d_a, d_b, d_d, cap, d_count, st, ws, js);
    const bool sparse = mode == 1;
    const int passes = sparse ? bdg::n_passes(t) : 1;
    const void* kern = sparse ? (t == 1 ? (const void*)bdg::sparse_tile_kernel<1, 0, false> : (const void*)bdg::sparse_tile_kernel<2, 0, false>)
                              : (t == 1 ? (const void*)bdg::edges_kernel<1> : t == 2 ? (const void*)bdg::edges_kernel<2>
                                                                                     : (const void*)bdg::edges_kernel<3>);
    int grid = 0;
    if (int rc = grid_for(kern, &grid, bdg::ENT)) return rc;
    if (const char* e = getenv("BDG_JOIN_CTAS")) grid = std::min(grid, ws->sms * std::max(1, atoi(e)));   // CTAs per SM of a join launch
    Plan plan;
    build_plan(N, part, nparts, grid * bdg::EW, plan, bdg::SB_MAX);
    const uint32_t n_items = plan.item_start.empty() ? 0 : plan.item_start.back();
    if (n_items == 0) return BDG_OK;
    const size_t nb_groups = plan.group_ids.size() * sizeof(uint32_t), nb_items = plan.item_start.size() * sizeof(uint32_t);
    const size_t hdr = PLAN_HDR * bdg::MAX_PASSES;
    if (int e = ws->plan.ensure(hdr + nb_groups + nb_items)) return e;
    char* d_plan = (char*)ws->plan.p;   // [headers | group_ids | item_start]
    CU_TRY(cudaMemsetAsync(d_plan, 0, hdr, st));
    for (int p = 0; p < bdg::MAX_PASSES; p++) ws->host_stats[p][0] = ws->host_stats[p][1] = 0;
    CU_TRY(cudaMemcpyAsync(d_plan + hdr, plan.group_ids.data(), nb_groups, cudaMemcpyHostToDevice, st));
    CU_TRY(cudaMemcpyAsync(d_plan + hdr + nb_groups, plan.item_start.data(), nb_items, cudaMemcpyHostToDevice, st));
    bdg::EdgeWork w;
    w.N = (uint32_t)N;
    w.t = t;
    w.T = bdg::qgram_threshold(t);
    w.group_ids = (const uint32_t*)(d_plan + hdr);
    w.item_start = (const uint32_t*)(d_plan + hdr + nb_groups);
    w.K = (uint32_t)plan.group_ids.size();
    w.n_items = n_items;
    w.chunk_cols = plan.chunk_cols;
    w.one = 1u;
    w.mone = 0xFFFFFFFFu;
    bdg::EdgeOut o{d_a, d_b, d_d, d_count, (unsigned long long)cap};
    const int blocks = (int)std::min<uint64_t>((uint64_t)grid, (n_items + bdg::EW - 1) / bdg::EW);
    // sparse passes are independent (disjoint outputs through one atomic cursor): pass 0 runs on the caller's stream, the others
    // on the device's auxiliary streams, so that one pass's sort / scan and its tail overlap the neighbour's tile kernel
    const bool fork = sparse && passes > 1 && !getenv("BDG_EDGE_SERIAL");
    cudaStream_t caller = st;
    if (fork) CU_TRY(cudaEventRecord(ws->ev_start, caller));
    for (int p = 0; p < passes; p++) {
        st = (fork && p > 0) ? ws->aux[p] : caller;
        if (fork && p > 0) CU_TRY(cudaStreamWaitEvent(st, ws->ev_start, 0));
        w.item_counter = (unsigned int*)(d_plan + PLAN_HDR * p);
        w.stats = (unsigned long long*)(d_plan + PLAN_HDR * p + HDR_STATS);
        w.pass = p;
        w.rot = sparse ? bdg::pass_rot(t, p) : 0;
        w.sorted = d_sorted;
        if (w.rot != 0) {   // this pass scans the array in the order of rotl(key, rot): rotate, radix-sort
            if (int e = ws->rot_in[p].ensure(N * 4)) return e;
            if (int e = ws->rot_sorted[p].ensure(N * 4)) return e;
            size_t tmp_bytes = 0;
            CU_TRY(cub::DeviceRadixSort::SortKeys(nullptr, tmp_bytes, (const uint32_t*)ws->rot_in[p].p, (uint32_t*)ws->rot_sorted[p].p, (int)N, 0, 32, st));
            if (int e = ws->sort_tmp[p].ensure(tmp_bytes)) return e;
            const int rb = (int)std::min<size_t>((N + 255) / 256, (size_t)ws->sms * 8);
            bdg::rotate_keys_kernel<<<rb, 256, 0, st>>>(d_sorted, (uint32_t*)ws->rot_in[p].p, (uint32_t)N, w.rot);
            g_launches++;
            CU_TRY(cub::DeviceRadixSort::SortKeys(ws->sort_tmp[p].p, tmp_bytes, (const uint32_t*)ws->rot_in[p].p, (uint32_t*)ws->rot_sorted[p].p, (int)N, 0, 32, st));
            w.sorted = (const uint32_t*)ws->rot_sorted[p].p;
        }
        if (!sparse) {
            if (t == 1) bdg::edges_kernel<1><<<blocks, bdg::ENT, 0, st>>>(w, o);
            else if (t == 2) bdg::edges_kernel<2><<<blocks, bdg::ENT, 0, st>>>(w, o);
            else bdg::edges_kernel<3><<<blocks, bdg::ENT, 0, st>>>(w, o);
        } else {
            // level 1: interval scan of every (owned row group, sub-tile right of it) -> compact tile list
            const uint32_t NS = (uint32_t)((N + bdg::SSB - 1) / bdg::SSB);
            if (int e = ws->tile_bnd[p].ensure((size_t)NS * sizeof(uint2))) return e;
            if (ws->tile_list[p].cap == 0) {
                size_t want = std::max<size_t>((size_t)1 << 22, 4 * N);
                if (const char* e = getenv("BDG_TILE_LIST_CAP")) want = (size_t)std::max(1ll, atoll(e));   // tests: force the regrow path
                if (int e = ws->tile_list[p].ensure(want * sizeof(uint2))) return e;
            }
            bdg::tile_bounds_kernel<<<std::min<uint32_t>((NS + 255) / 256, (uint32_t)ws->sms * 8), 256, 0, st>>>(w.sorted, w.N, (uint2*)ws->tile_bnd[p].p, NS);
            g_launches++;
            // no read-back between the scan and the tile kernel: the tile kernel reads the list length on the device and, if
            // the list was too small, poisons the edge count (bit 63), which every caller inspects before using the edges
            bdg::TileList l{(uint2*)ws->tile_list[p].p, (unsigned long long*)(d_plan + PLAN_HDR * p + HDR_LIST), ws->tile_list[p].cap / sizeof(uint2)};
            const int sblocks = (int)std::min<uint64_t>(w.K, (uint64_t)ws->sms * 16);
            BDG_PASS_DISPATCH(launch_scan, sblocks, st, w, (const uint2*)ws->tile_bnd[p].p, NS, l);
            g_launches++;
            CU_TRY(cudaGetLastError());
            uint64_t tests = 0;
            for (uint32_t g : plan.group_ids) tests += NS - std::min<uint64_t>(NS, (uint64_t)g * (bdg::GROUP / bdg::SSB));
            ws->host_stats[p][0] = tests;
            BDG_PASS_DISPATCH(launch_tiles, grid, st, w, o, l);
        }
        g_launches++;
        CU_TRY(cudaGetLastError());
        if (fork && p > 0) CU_TRY(cudaEventRecord(ws->ev_done[p], st));
    }
    if (fork)
        for (int p = 1; p < passes; p++) CU_TRY(cudaStreamWaitEvent(caller, ws->ev_done[p], 0));
    return BDG_OK;
}


// Q x W scoring through the sparse machinery (max_d <= 2): queries and targets are each sorted by the pass's rotated
// key (original indices ride along), tiles of (256 queries x 128 targets) whose key intervals cannot meet are decided
// by the scan, the rest get the quick test, survivors the exact plain distance and an atomicMin on the query's key.
int launch_nearest_sparse(const uint32_t* d_q, size_t Q, const uint32_t* d_t, size_t W, int max_d, uint32_t* d_keys, cudaStream_t st, DevCtx* ws)
{
    const int T_ = max_d <= 1 ? 1 : 2;
    const int passes = bdg::n_passes(T_);
    for (Buf* b : {&ws->nn_q.key, &ws->nn_q.pay, &ws->nn_q.key_sorted, &ws->nn_q.pay_sorted}) if (int e = b->ensure(Q * 4)) return e;
    for (Buf* b : {&ws->nn_t.key, &ws->nn_t.pay, &ws->nn_t.key_sorted, &ws->nn_t.pay_sorted}) if (int e = b->ensure(W * 4)) return e;
    uint32_t *qk = (uint32_t*)ws->nn_q.key.p, *qp = (uint32_t*)ws->nn_q.pay.p, *qks = (uint32_t*)ws->nn_q.key_sorted.p, *qps = (uint32_t*)ws->nn_q.pay_sorted.p;
    uint32_t *tk = (uint32_t*)ws->nn_t.key.p, *tp = (uint32_t*)ws->nn_t.pay.p, *tks = (uint32_t*)ws->nn_t.key_sorted.p, *tps = (uint32_t*)ws->nn_t.pay_sorted.p;
    size_t tmp_q = 0, tmp_t = 0;
    CU_TRY(cub::DeviceRadixSort::SortPairs(nullptr, tmp_q, qk, qks, qp, qps, (int)Q, 0, 32, st));
    CU_TRY(cub::DeviceRadixSort::SortPairs(nullptr, tmp_t, tk, tks, tp, tps, (int)W, 0, 32, st));
    if (int e = ws->nn_tmp.ensure(std::max(tmp_q, tmp_t))) return e;
    const uint32_t NS = (uint32_t)((W + bdg::SSB - 1) / bdg::SSB);
    const uint32_t K = (uint32_t)((Q + bdg::GROUP - 1) / bdg::GROUP);
    if (int e = ws->tile_bnd[0].ensure((size_t)NS * sizeof(uint2))) return e;
    if (ws->tile_list[0].cap == 0)
        if (int e = ws->tile_list[0].ensure(((size_t)1 << 22) * sizeof(uint2))) return e;
    if (int e = ws->plan.ensure(PLAN_HDR * bdg::MAX_PASSES)) return e;
    char* d_plan = (char*)ws->plan.p;   // only the headers are used here; a cached edge plan behind them stays valid
    CU_TRY(cudaMemsetAsync(d_plan, 0, PLAN_HDR * bdg::MAX_PASSES, st));
    int grid = 0;
    if (int rc = grid_for(T_ == 1 ? (const void*)bdg::sparse_tile_kernel<1, 0, true> : (const void*)bdg::sparse_tile_kernel<2, 0, true>, &grid, bdg::ENT)) return rc;
    const int t = T_;   // BDG_PASS_DISPATCH reads `t` and `p`
    for (int p = 0; p < passes; p++) {
        const int rot = bdg::pass_rot(T_, p);
        const int qb = (int)std::min<size_t>((Q + 255) / 256, (size_t)ws->sms * 8), tb = (int)std::min<size_t>((W + 255) / 256, (size_t)ws->sms * 8);
        bdg::rotate_keys_iota_kernel<<<qb, 256, 0, st>>>(d_q, qk, qp, (uint32_t)Q, rot);
        bdg::rotate_keys_iota_kernel<<<tb, 256, 0, st>>>(d_t, tk, tp, (uint32_t)W, rot);
        CU_TRY(cub::DeviceRadixSort::SortPairs(ws->nn_tmp.p, tmp_q, qk, qks, qp, qps, (int)Q, 0, 32, st));
        CU_TRY(cub::DeviceRadixSort::SortPairs(ws->nn_tmp.p, tmp_t, tk, tks, tp, tps, (int)W, 0, 32, st));
        bdg::tile_bounds_kernel<<<std::min<uint32_t>((NS + 255) / 256, (uint32_t)ws->sms * 8), 256, 0, st>>>(tks, (uint32_t)W, (uint2*)ws->tile_bnd[0].p, NS);
        g_launches += 3;
        bdg::EdgeWork w{};
        w.sorted = qks; w.N = (uint32_t)Q; w.t = max_d; w.T = 0; w.group_ids = nullptr; w.item_start = nullptr; w.K = K;
        w.item_counter = (unsigned int*)(d_plan + PLAN_HDR * p);
        w.stats = nullptr; w.one = 1u; w.mone = 0xFFFFFFFFu; w.pass = p; w.rot = rot;
        w.cols = tks; w.NC = (uint32_t)W; w.row_pay = qps; w.col_pay = tps; w.near_keys = d_keys;
        unsigned long long n_tiles = 0;
        for (int attempt = 0; attempt < 2; attempt++) {
            bdg::TileList l{(uint2*)ws->tile_list[0].p, (unsigned long long*)(d_plan + PLAN_HDR * p + HDR_LIST), ws->tile_list[0].cap / sizeof(uint2)};
            CU_TRY(cudaMemsetAsync(l.count, 0, 8, st));
            const int sblocks = (int)std::min<uint64_t>(K, (uint64_t)ws->sms * 16);
            BDG_PASS_DISPATCH(launch_scan_bip, sblocks, st, w, (const uint2*)ws->tile_bnd[0].p, NS, l);
            g_launches++;
            CU_TRY(cudaGetLastError());
            CU_TRY(cudaMemcpyAsync(&n_tiles, l.count, 8, cudaMemcpyDeviceToHost, st));
            CU_TRY(cudaStreamSynchronize(st));
            if (n_tiles <= l.cap) break;
            if (attempt == 1) return fail(BDG_ERR_CUDA, "tile list count changed between identical scans");
            if (int e = ws->tile_list[0].ensure((size_t)n_tiles * sizeof(uint2))) return e;
        }
        if (n_tiles == 0) continue;
        bdg::TileList l{(uint2*)ws->tile_list[0].p, (unsigned long long*)(d_plan + PLAN_HDR * p + HDR_LIST), ws->tile_list[0].cap / sizeof(uint2)};
        const int tblocks = (int)std::min<uint64_t>((uint64_t)grid, (n_tiles + bdg::EW - 1) / bdg::EW);
        bdg::EdgeOut o{nullptr, nullptr, nullptr, nullptr, 0};
        BDG_PASS_DISPATCH(launch_tiles_bip, tblocks, st, w, o, l);
        g_launches++;
        CU_TRY(cudaGetLastError());
    }
    return BDG_OK;
}

DevCtx* ctx_of_current_device();

DevCtx* ctx_of_current_device()
{
    int dev = -1;
    if (cudaGetDevice(&dev) != cudaSuccess) return nullptr;
    for (auto& c : g_ctx) if (c.dev == dev) return &c;
    return nullptr;
}

int need_ctx()
{
    if (g_ctx.empty()) {
        int rc = bdg_init(nullptr, 0);
        if (rc) return rc;
    }
    return BDG_OK;
}

// The first claimed context, its device made current, when `token` names the read map live there.
int map_ctx(unsigned long long token, DevCtx** out)
{
    if (int rc = need_ctx()) return rc;
    DevCtx& c = g_ctx[0];
    if (token == 0 || token != c.map.token) return fail(BDG_ERR_ARG, "stale read-map token: a later dedup call has reused the workspaces");
    CU_TRY(cudaSetDevice(c.dev));
    *out = &c;
    return BDG_OK;
}

// The per-pass headers of the last edge launch on c (PLAN_HDR bytes each: work cursor, tile-list count, statistics), read back on st.
constexpr size_t PLAN_WORDS = (PLAN_HDR / 8) * bdg::MAX_PASSES;
int read_plan_headers(const DevCtx* c, cudaStream_t st, unsigned long long (&v)[PLAN_WORDS])
{
    if (!c || !c->plan.p) return fail(BDG_ERR_ARG, "no edge launch on this device yet");
    CU_TRY(cudaMemcpyAsync(v, c->plan.p, sizeof(v), cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaStreamSynchronize(st));
    return BDG_OK;
}

// After an edge count that came back with bit 63 set (a sparse pass listed more tiles than its list holds): every pass's tile
// list grows to the longest list any pass asked for, so that the launch can run again.
int grow_tile_lists(DevCtx& c)
{
    unsigned long long v[PLAN_WORDS];
    if (int rc = read_plan_headers(&c, c.stream, v)) return rc;
    unsigned long long need = 0;
    for (int p = 0; p < bdg::MAX_PASSES; p++) need = std::max(need, v[(PLAN_HDR / 8) * p + HDR_LIST / 8]);
    for (int p = 0; p < bdg::MAX_PASSES; p++)
        if (int e = c.tile_list[p].ensure((size_t)need * sizeof(uint2))) return e;
    return BDG_OK;
}

int check_sorted(const uint32_t* v, size_t N)
{
    for (size_t i = 1; i < N; i++)
        if (v[i] <= v[i - 1]) return fail(BDG_ERR_ARG, "input not strictly increasing at index %zu", i);
    return BDG_OK;
}

size_t edge_cap_guess(size_t N, int t, int nparts)
{
    // a too small guess costs a whole second run (the kernel only counts what it cannot store); 9 bytes per slot are cheap
    size_t per_row = t <= 1 ? 16 : 64;
    if (const char* e = getenv("BDG_EDGE_CAP_PER_ROW")) per_row = (size_t)std::max(1ll, atoll(e));
    return std::max<size_t>(1u << 16, per_row * N / (size_t)nparts + 1024);
}

// The bdg_dev_* forms of the correction step read and write caller memory on the first claimed device, where the read map lives.
int check_on_first(const void* p, const char* what)
{
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        (void)cudaGetLastError();
        return fail(BDG_ERR_ARG, "%s is not a CUDA pointer", what);
    }
    if ((a.type != cudaMemoryTypeDevice && a.type != cudaMemoryTypeManaged) || a.device != g_ctx[0].dev)
        return fail(BDG_ERR_ARG, "%s is not memory of device %d (the first claimed device)", what, g_ctx[0].dev);
    return BDG_OK;
}

// Stream order of a bdg_dev_* call that runs on the library's stream of the first device: begin() holds that stream until the
// work the caller queued on its own stream so far is done (it produces the inputs and frees the output buffers); the
// destructor, on every return path, holds the caller's stream until the library's work is done (it writes the outputs and
// reads the inputs).
// A host-buffer call passes the library's own stream: there is nothing to order.
struct CallerOrder {
    DevCtx& c;
    cudaStream_t caller;
    bool armed = false;
    CallerOrder(DevCtx& c_, void* stream) : c(c_), caller((cudaStream_t)stream) {}
    int begin()
    {
        if (caller == c.stream) return BDG_OK;
        CU_TRY(cudaEventRecord(c.ev_caller, caller));
        CU_TRY(cudaStreamWaitEvent(c.stream, c.ev_caller, 0));
        armed = true;
        return BDG_OK;
    }
    ~CallerOrder()
    {
        if (armed && cudaEventRecord(c.ev_caller, c.stream) == cudaSuccess) cudaStreamWaitEvent(caller, c.ev_caller, 0);
    }
};

// The correction step runs on the first claimed context; its device is made current.
int first_ctx(DevCtx** out)
{
    if (int rc = need_ctx()) return rc;
    *out = &g_ctx[0];
    CU_TRY(cudaSetDevice(g_ctx[0].dev));
    return BDG_OK;
}

// What the argument check of an entry point returns when the call has nothing to do (an empty input); the entry point then
// returns BDG_OK (every error code is negative).
constexpr int EMPTY = 1;
int done(int rc) { return rc == EMPTY ? BDG_OK : rc; }

// c.io carved into consecutive pieces (256-byte aligned), grown first to their sum: the uploads, outputs and per-read scratch of
// one call.  Every call that stages there ends with a synchronise or runs in stream order on c.stream, so the next call finds
// it free.  Example: stage(c, {piece(d_q, Q * 4), piece(d_hit, Q)}).
struct Piece { void** at; size_t bytes; };
template <typename T> Piece piece(T*& p, size_t bytes) { return {(void**)&p, bytes}; }

int stage(DevCtx& c, std::initializer_list<Piece> parts)
{
    auto round = [](size_t b) { return (b + 255) / 256 * 256; };
    size_t total = 0;
    for (const Piece& x : parts) total += round(x.bytes);
    if (int e = c.io.ensure(std::max<size_t>(total, 1))) return e;
    char* at = (char*)c.io.p;
    for (const Piece& x : parts) { *x.at = at; at += round(x.bytes); }
    return BDG_OK;
}

// The sort check of a whitelist on the device: sort_check launches it on c.stream, sort_check_result reads the index of the first
// entry that is not above its predecessor back (waiting for everything queued on c.stream) and refuses the whitelist if there is one.
int sort_check(DevCtx& c, const uint32_t* d_wl, size_t W)
{
    if (int e = c.sort_flag.ensure(8)) return e;
    CU_TRY(cudaMemsetAsync(c.sort_flag.p, 0xFF, 8, c.stream));
    if (W > 1) {
        bdg::sorted_check_kernel<false><<<(int)std::min<size_t>((W + 255) / 256, (size_t)c.sms * 8), 256, 0, c.stream>>>(
            d_wl, (uint32_t)W, (unsigned long long*)c.sort_flag.p);
        g_launches++;
    }
    CU_TRY(cudaGetLastError());
    return BDG_OK;
}

int sort_check_result(DevCtx& c)
{
    unsigned long long first_bad = ~0ull;
    CU_TRY(cudaMemcpyAsync(&first_bad, c.sort_flag.p, 8, cudaMemcpyDeviceToHost, c.stream));
    CU_TRY(cudaStreamSynchronize(c.stream));
    if (first_bad != ~0ull) return fail(BDG_ERR_ARG, "whitelist not sorted at index %llu", first_bad);
    return BDG_OK;
}

}  // namespace

// Handle of one edge construction: the edges stay in the devices' grow-only workspaces until the caller copies them
// out (bdg_edges_copy: ONE device-to-host copy per array, straight into the caller's buffers).  A later build on the
// same device reuses those workspaces, which makes older handles stale (checked through the generation numbers).
struct bdg_edges {
    std::vector<int> ctx;                 // indices into g_ctx
    std::vector<size_t> count;            // edges held by each of them
    std::vector<unsigned long long> gen;  // workspace generation at build time
    unsigned long long read_map = 0;       // token of the read map whose ascending array the edges were built from (0: a caller's array)
};

// Known strings of a KmerIndexer / QGramIndex, resident on one device, plus grow-only query / result buffers.
struct bdg_kmer_index {
    int dev = -1;
    size_t W = 0;
    Buf wl;
    Buf hit_q, hit_w, hit_cnt;        // host-buffer queries: the hits before they are copied out
    Buf mult;                         // packed 6-mer positions per hit (the device form unpacks them)
    Buf total;                        // hit counter
    Buf kstart, post, scratch;       // posting lists: first posting of every 6-mer (4097 words), string ids grouped by 6-mer
    bool posted = false;
    cudaEvent_t ev[2] = {nullptr, nullptr};   // around the last query's kernel
    bool timed = false;
};

extern "C" {

const char* bdg_version(void) { return "badger_b200 0.1 (sm_100a)"; }
const char* bdg_last_error(void) { return g_err; }
int bdg_device_count(void) { return (int)g_ctx.size(); }
unsigned long long bdg_launch_count(void) { return g_launches.load(); }

int bdg_init(const int* device_ids, int n_devices)
{
    int visible = 0;
    cudaError_t e = cudaGetDeviceCount(&visible);
    if (e != cudaSuccess || visible == 0)
        return fail(BDG_ERR_NODEVICE, "no CUDA device: %s (libbadger_b200 has no CPU fallback)",
                    e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
    std::vector<int> ids;
    if (!device_ids || n_devices <= 0) for (int i = 0; i < visible; i++) ids.push_back(i);
    else ids.assign(device_ids, device_ids + n_devices);
    bool same = ids.size() == g_ctx.size();
    for (size_t i = 0; same && i < ids.size(); i++) same = g_ctx[i].dev == ids[i];
    if (same) return BDG_OK;
    bdg_shutdown();
    for (int id : ids) {
        if (id < 0 || id >= visible) { bdg_shutdown(); return fail(BDG_ERR_ARG, "device id %d out of range (%d visible)", id, visible); }
        DevCtx c;
        c.dev = id;
        CU_TRY(cudaSetDevice(id));
        cudaDeviceProp prop;
        CU_TRY(cudaGetDeviceProperties(&prop, id));
        if (prop.major < 10) { bdg_shutdown(); return fail(BDG_ERR_NODEVICE, "device %d is sm_%d%d; this library is built for sm_100a only", id, prop.major, prop.minor); }
        c.sms = prop.multiProcessorCount;
        CU_TRY(cudaStreamCreateWithFlags(&c.stream, cudaStreamNonBlocking));
        CU_TRY(cudaEventCreateWithFlags(&c.ev_start, cudaEventDisableTiming));
        CU_TRY(cudaEventCreateWithFlags(&c.ev_caller, cudaEventDisableTiming));
        for (int p = 1; p < bdg::MAX_PASSES; p++) {
            CU_TRY(cudaStreamCreateWithFlags(&c.aux[p], cudaStreamNonBlocking));
            CU_TRY(cudaEventCreateWithFlags(&c.ev_done[p], cudaEventDisableTiming));
        }
        g_ctx.push_back(std::move(c));
    }
    // direct NVLink copies into the first device (bdg_cluster_levels_from_edges gathers the other devices' edge lists there);
    // without peer access cudaMemcpyPeerAsync stages through host memory
    // (both directions: the edge lists travel to the first device, the distinct-barcode array fans out from it)
    for (size_t g = 1; g < g_ctx.size(); g++) {
        for (int dir = 0; dir < 2; dir++) {
            const int from = dir ? g_ctx[g].dev : g_ctx[0].dev, to = dir ? g_ctx[0].dev : g_ctx[g].dev;
            int can = 0;
            CU_TRY(cudaSetDevice(from));
            if (cudaDeviceCanAccessPeer(&can, from, to) == cudaSuccess && can) {
                const cudaError_t pe = cudaDeviceEnablePeerAccess(to, 0);
                if (pe != cudaSuccess) (void)cudaGetLastError();      // already enabled (e.g. by the caller's framework): fine
            }
        }
    }
    CU_TRY(cudaSetDevice(g_ctx[0].dev));
    return BDG_OK;
}

void bdg_shutdown(void)
{
    while (!g_ctx.empty()) {
        DevCtx& c = g_ctx.back();
        cudaSetDevice(c.dev);                              // the context's buffers are freed on its device
        if (c.stream) { cudaStreamSynchronize(c.stream); cudaStreamDestroy(c.stream); }
        for (int p = 0; p < bdg::MAX_PASSES; p++) {
            if (c.aux[p]) cudaStreamDestroy(c.aux[p]);
            if (c.ev_done[p]) cudaEventDestroy(c.ev_done[p]);
        }
        if (c.ev_start) cudaEventDestroy(c.ev_start);
        if (c.ev_caller) cudaEventDestroy(c.ev_caller);
        if (c.snap_host) { cudaFreeHost(c.snap_host); c.snap_host = nullptr; for (auto& e : c.ev_snap) if (e) cudaEventDestroy(e);
                           for (int q = 0; q < 2; q++) { if (c.ev_pre[q]) cudaEventDestroy(c.ev_pre[q]); if (c.ev_join[q]) cudaEventDestroy(c.ev_join[q]); } }
        g_ctx.pop_back();
    }
}

unsigned long long bdg_part_pairs(size_t N, int part, int nparts)
{
    if (nparts < 1 || part < 0 || part >= nparts) return 0;
    Plan p;
    build_plan(N, part, nparts, 1, p);
    return p.pairs;
}

// ---------------------------------------------------------------- device-resident entry points
int bdg_dev_edges_build(const uint32_t* d_sorted, size_t N, int t, int part, int nparts, uint32_t* d_a, uint32_t* d_b,
                        uint8_t* d_d, size_t cap, unsigned long long* d_count, void* stream)
{
    if (!d_count || (N && !d_sorted) || (cap && (!d_a || !d_b || !d_d))) return fail(BDG_ERR_ARG, "NULL pointer argument");
    DevCtx* c = ctx_of_current_device();
    return launch_edges(d_sorted, N, t, part, nparts, d_a, d_b, d_d, cap, d_count, (cudaStream_t)stream, c);
}

// Page-locked host memory for callers that want device-to-host copies at full PCIe speed (badger_b200.ops keeps a small
// pool of such blocks behind the numpy arrays it returns).
int bdg_host_alloc(size_t bytes, void** out)
{
    if (!out) return fail(BDG_ERR_ARG, "NULL pointer argument");
    *out = nullptr;
    if (int rc = need_ctx()) return rc;
    cudaError_t e = cudaHostAlloc(out, std::max<size_t>(bytes, 1), cudaHostAllocPortable);
    if (e != cudaSuccess) { *out = nullptr; return fail(BDG_ERR_OOM, "cudaHostAlloc of %zu bytes: %s", bytes, cudaGetErrorString(e)); }
    return BDG_OK;
}

void bdg_host_free(void* p)
{
    if (p) cudaFreeHost(p);
}

int bdg_set_edge_mode(int mode)
{
    if (mode < -1 || mode > 2) return fail(BDG_ERR_ARG, "edge mode must be -1 (default), 0 (dense), 1 (sparse) or 2 (join)");
    g_edge_mode = mode;
    return BDG_OK;
}

int bdg_dev_edges_stats(unsigned long long* out5, void* stream)
{
    if (!out5) return fail(BDG_ERR_ARG, "NULL pointer argument");
    DevCtx* c = ctx_of_current_device();
    unsigned long long v[PLAN_WORDS];
    if (int rc = read_plan_headers(c, (cudaStream_t)stream, v)) return rc;
    for (int k = 0; k < 5; k++) {
        out5[k] = 0;
        const int slot = k < 4 ? k : 7;
        for (int p = 0; p < bdg::MAX_PASSES; p++) {
            out5[k] += v[(PLAN_HDR / 8) * p + HDR_STATS / 8 + slot];
            if (k == 0) out5[k] += c->host_stats[p][0];                       // interval tests of the sparse scans (counted on the host)
            if (k == 1) out5[k] += v[(PLAN_HDR / 8) * p + HDR_LIST / 8];      // tiles the scans listed
        }
    }
    return BDG_OK;
}

// The kernels' eight raw counters summed over the passes (join form: [0] work units, [2] pairs tested, [3] candidates,
// [6] candidates with D <= 2, [7] pairs whose 6-mer score was computed; [4] / [5] sum / max of the warps' busy time in ns).
int bdg_dev_edges_stats_raw(unsigned long long* out8, void* stream)
{
    if (!out8) return fail(BDG_ERR_ARG, "NULL pointer argument");
    unsigned long long v[PLAN_WORDS];
    if (int rc = read_plan_headers(ctx_of_current_device(), (cudaStream_t)stream, v)) return rc;
    for (int k = 0; k < 8; k++) {
        out8[k] = 0;
        for (int p = 0; p < bdg::MAX_PASSES; p++) {
            const unsigned long long x = v[(PLAN_HDR / 8) * p + HDR_STATS / 8 + k];
            out8[k] = k == 5 ? std::max(out8[k], x) : out8[k] + x;
        }
    }
    return BDG_OK;
}

// Development aid (tools/join_lane_stats.py): the lane-use counters of the join kernel (bdg_join.cuh g_join_lane), only in a build
// with -DBDG_JOIN_LANE_STATS; summed over every join launch on the current device since the last reset.
int bdg_join_lane_stats(unsigned long long* out8, int reset)
{
    if (!out8) return fail(BDG_ERR_ARG, "NULL pointer argument");
#ifdef BDG_JOIN_LANE_STATS
    CU_TRY(cudaDeviceSynchronize());
    CU_TRY(cudaMemcpyFromSymbol(out8, bdg::g_join_lane, 8 * sizeof(unsigned long long)));
    if (reset) {
        const unsigned long long zero[8] = {};
        CU_TRY(cudaMemcpyToSymbol(bdg::g_join_lane, zero, sizeof(zero)));
    }
    return BDG_OK;
#else
    (void)reset;
    return fail(BDG_ERR_UNSUPPORTED, "built without the join lane counters (make EXTRA=-DBDG_JOIN_LANE_STATS)");
#endif
}

// Development aid (tools/sweep_edges.py): per pass, sum and max over warps of the warp's exit time in ns
// measured from the first warp's start - the load-balance picture of the last edge launch.
int bdg_dev_edges_balance(unsigned long long* out /* 2 * MAX_PASSES */, void* stream)
{
    if (!out) return fail(BDG_ERR_ARG, "NULL pointer argument");
    unsigned long long v[PLAN_WORDS];
    if (int rc = read_plan_headers(ctx_of_current_device(), (cudaStream_t)stream, v)) return rc;
    for (int p = 0; p < bdg::MAX_PASSES; p++) {
        out[2 * p] = v[(PLAN_HDR / 8) * p + HDR_STATS / 8 + 4];
        out[2 * p + 1] = v[(PLAN_HDR / 8) * p + HDR_STATS / 8 + 5];
    }
    return BDG_OK;
}

int bdg_dev_pack16(const char* d_seqs, size_t R, uint32_t* d_out, uint8_t* d_valid, void* stream)
{
    if (R == 0) return BDG_OK;
    if (!d_seqs || !d_out || !d_valid) return fail(BDG_ERR_ARG, "NULL pointer argument");
    if ((uintptr_t)d_seqs % 16) return fail(BDG_ERR_ARG, "sequence buffer must be 16-byte aligned");
    int grid = 0;
    if (int rc = grid_for((const void*)bdg::pack16_kernel, &grid)) return rc;
    const int blocks = (int)std::min<uint64_t>((uint64_t)grid, (R + 4 * bdg::NT - 1) / (4 * bdg::NT));
    bdg::pack16_kernel<<<blocks, bdg::NT, 0, (cudaStream_t)stream>>>((const uint4*)d_seqs, R, d_out, d_valid);
    g_launches++;
    CU_TRY(cudaGetLastError());
    return BDG_OK;
}

static int member_sorted_args(const uint32_t* wl, size_t W, const uint32_t* q, size_t Q, const uint8_t* hit)
{
    if (Q == 0) return EMPTY;
    if (!q || !hit || (W && !wl)) return fail(BDG_ERR_ARG, "NULL pointer argument");
    if (W > 0xFFFFFFFFull || Q > 0xFFFFFFFFull) return fail(BDG_ERR_ARG, "size exceeds 2^32");
    return BDG_OK;
}

// Membership of Q > 0 queries in the sorted whitelist, on the current device and the given stream.
static int member_sorted_body(const uint32_t* d_wl, size_t W, const uint32_t* d_q, size_t Q, uint8_t* d_hit, cudaStream_t st)
{
    if (W == 0) { CU_TRY(cudaMemsetAsync(d_hit, 0, Q, st)); return BDG_OK; }
    int grid = 0;
    if (int rc = grid_for((const void*)bdg::member_kernel, &grid)) return rc;
    const int blocks = (int)std::min<uint64_t>((uint64_t)grid, (Q + bdg::NT - 1) / bdg::NT);
    bdg::member_kernel<<<blocks, bdg::NT, 0, st>>>(d_wl, (uint32_t)W, d_q, (uint32_t)Q, d_hit);
    g_launches++;
    CU_TRY(cudaGetLastError());
    return BDG_OK;
}

int bdg_dev_member_sorted(const uint32_t* d_wl, size_t W, const uint32_t* d_q, size_t Q, uint8_t* d_hit, void* stream)
{
    if (int rc = member_sorted_args(d_wl, W, d_q, Q, d_hit)) return done(rc);
    return member_sorted_body(d_wl, W, d_q, Q, d_hit, (cudaStream_t)stream);
}

int bdg_dev_nearest_bounded(const uint32_t* d_q, size_t Q, const uint32_t* d_t, size_t W, int max_d, uint32_t* d_keys,
                            int32_t* d_argmin, uint8_t* d_dist, void* stream)
{
    if (Q == 0) return BDG_OK;
    if (!d_q || !d_keys || !d_argmin || !d_dist || (W && !d_t)) return fail(BDG_ERR_ARG, "NULL pointer argument");
    if (W >= (1ull << bdg::NEAR_IDX_BITS) || Q > 0xFFFFFFFFull) return fail(BDG_ERR_ARG, "W must be < 2^28 and Q < 2^32");
    if (max_d > 15) return fail(BDG_ERR_ARG, "max_d must be <= 15 (a distance of 16 does not fit the packed (distance, index) key)");
    cudaStream_t st = (cudaStream_t)stream;
    CU_TRY(cudaMemsetAsync(d_keys, 0xFF, Q * sizeof(uint32_t), st));
    DevCtx* ws = ctx_of_current_device();
    const bool sparse = ws && W > 0 && max_d >= 0 && max_d <= 2 && (unsigned long long)Q * W >= (1ull << 24) && !getenv("BDG_NEAREST_DENSE");
    if (sparse) {
        if (int rc = launch_nearest_sparse(d_q, Q, d_t, W, max_d, d_keys, st, ws)) return rc;
    } else if (W > 0 && max_d >= 0) {
        int sms = 0, dev = 0;
        CU_TRY(cudaGetDevice(&dev));
        CU_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        const uint32_t gx = (uint32_t)((Q + bdg::ROW_TILE - 1) / bdg::ROW_TILE);
        uint32_t gy = std::max<uint32_t>(1, (uint32_t)(4 * sms) / gx);          // split targets when there are few query tiles
        gy = std::min<uint32_t>(gy, (uint32_t)((W + bdg::NEAR_TB - 1) / bdg::NEAR_TB));
        gy = std::min<uint32_t>(gy, 65535u);
        uint32_t wpb = (uint32_t)((W + gy - 1) / gy);
        wpb = (wpb + bdg::NEAR_TB - 1) / bdg::NEAR_TB * bdg::NEAR_TB;
        gy = (uint32_t)((W + wpb - 1) / wpb);
        dim3 grid(gx, gy);
        if (max_d <= 2) bdg::nearest_kernel<true><<<grid, bdg::NT, 0, st>>>(d_q, (uint32_t)Q, d_t, (uint32_t)W, max_d, wpb, d_keys);
        else bdg::nearest_kernel<false><<<grid, bdg::NT, 0, st>>>(d_q, (uint32_t)Q, d_t, (uint32_t)W, max_d, wpb, d_keys);
        g_launches++;
        CU_TRY(cudaGetLastError());
    }
    bdg::nearest_finish_kernel<<<(unsigned)((Q + 255) / 256), 256, 0, st>>>(d_keys, (uint32_t)Q, d_argmin, d_dist);
    g_launches++;
    CU_TRY(cudaGetLastError());
    return BDG_OK;
}

int bdg_dev_pipe_probe(int kind, int blocks, int iters, uint32_t* d_sink, unsigned long long* ops_per_thread, void* stream)
{
    if (!d_sink || blocks < 1 || iters < 1) return fail(BDG_ERR_ARG, "bad probe arguments");
    cudaStream_t st = (cudaStream_t)stream;
    switch (kind) {
    case 0: bdg::pipe_probe_kernel<0><<<blocks, bdg::NT, 0, st>>>(iters, d_sink); break;
    case 1: bdg::pipe_probe_kernel<1><<<blocks, bdg::NT, 0, st>>>(iters, d_sink); break;
    case 2: bdg::pipe_probe_kernel<2><<<blocks, bdg::NT, 0, st>>>(iters, d_sink); break;
    case 3: bdg::pipe_probe_kernel<3><<<blocks, bdg::NT, 0, st>>>(iters, d_sink); break;
    default: return fail(BDG_ERR_ARG, "unknown probe kind %d", kind);
    }
    g_launches++;
    CU_TRY(cudaGetLastError());
    if (ops_per_thread) *ops_per_thread = 64ull * (unsigned long long)iters;
    return BDG_OK;
}

// ---------------------------------------------------------------- host-buffer entry points
// ---- a-2  dedup + count in first-seen order (barcode_graph.py:192-204) ------------------------------------
// The keys of the n reads sit in dd[0] (ReadMap::keys) on entry (put there by the caller).  On return dd[] holds the arrays
// ReadMap names; keep_map: compute the read -> first-seen position map and leave it in dd[7] (download it too when
// read_to_distinct != NULL).
static int dedup_core(DevCtx& c, uint32_t n, uint32_t* distinct, uint32_t* counts, uint32_t* read_to_distinct, uint32_t* sorted_pos,
                      bool keep_map, size_t* n_distinct, uint32_t* sorted_distinct = nullptr)
{
    cudaStream_t st = c.stream;
    Buf* dd = c.map.dd;
    const size_t R = n;
    // dd[0] keys, [1] idx, [2] sorted keys, [3] sorted idx, [4] heads, [5] inclusive scan, [6] run key, [7] run first, [8] run start, [9] scratch
    for (int k = 1; k < 9; k++) if (int e = dd[k].ensure(R * 4)) return e;
    uint32_t *d_k = (uint32_t*)dd[0].p, *d_i = (uint32_t*)dd[1].p, *d_sk = (uint32_t*)dd[2].p, *d_si = (uint32_t*)dd[3].p;
    uint32_t *d_head = (uint32_t*)dd[4].p, *d_scan = (uint32_t*)dd[5].p, *d_rk = (uint32_t*)dd[6].p, *d_rf = (uint32_t*)dd[7].p, *d_rs = (uint32_t*)dd[8].p;
    size_t tmp1 = 0, tmp2 = 0;
    CU_TRY(cub::DeviceRadixSort::SortPairs(nullptr, tmp1, d_k, d_sk, d_i, d_si, (int)n, 0, 32, st));
    CU_TRY(cub::DeviceScan::InclusiveSum(nullptr, tmp2, d_head, d_scan, (int)n, st));
    if (int e = dd[9].ensure(std::max(tmp1, tmp2))) return e;
    const int blocks = (int)std::min<size_t>((R + 255) / 256, (size_t)c.sms * 8);
    bdg::iota_kernel<<<blocks, 256, 0, st>>>(d_i, n);
    CU_TRY(cub::DeviceRadixSort::SortPairs(dd[9].p, tmp1, d_k, d_sk, d_i, d_si, (int)n, 0, 32, st));
    bdg::dedup_heads_kernel<<<blocks, 256, 0, st>>>(d_sk, n, d_head);
    CU_TRY(cub::DeviceScan::InclusiveSum(dd[9].p, tmp2, d_head, d_scan, (int)n, st));
    bdg::dedup_runs_kernel<<<blocks, 256, 0, st>>>(d_sk, d_si, d_head, d_scan, n, d_rk, d_rf, d_rs);
    uint32_t n_runs = 0;
    CU_TRY(cudaMemcpyAsync(&n_runs, d_scan + (n - 1), 4, cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaStreamSynchronize(st));
    g_launches += 3;
    // order the runs by their first read index: reuse keys/idx buffers (d_k := sorted first indices, d_i := order), heads := iota
    bdg::iota_kernel<<<blocks, 256, 0, st>>>(d_head, n_runs);
    CU_TRY(cub::DeviceRadixSort::SortPairs(dd[9].p, tmp1, d_rf, d_k, d_head, d_i, (int)n_runs, 0, 32, st));
    // d_sk is free again after dedup_runs: distinct / counts / pos_of_run live in d_sk, d_k, d_head
    uint32_t *d_distinct = d_sk, *d_counts = d_k, *d_pos = d_head;
    bdg::dedup_finish_kernel<<<blocks, 256, 0, st>>>(d_i, d_rk, d_rs, n_runs, n, d_distinct, d_counts, d_pos);
    g_launches += 2;
    if (distinct) CU_TRY(cudaMemcpyAsync(distinct, d_distinct, (size_t)n_runs * 4, cudaMemcpyDeviceToHost, st));
    if (counts) CU_TRY(cudaMemcpyAsync(counts, d_counts, (size_t)n_runs * 4, cudaMemcpyDeviceToHost, st));
    if (sorted_pos) CU_TRY(cudaMemcpyAsync(sorted_pos, d_i, (size_t)n_runs * 4, cudaMemcpyDeviceToHost, st));   // order[pos] = run = ascending position
    if (sorted_distinct) CU_TRY(cudaMemcpyAsync(sorted_distinct, d_rk, (size_t)n_runs * 4, cudaMemcpyDeviceToHost, st));   // runs are numbered in key order
    if (keep_map || read_to_distinct) {
        bdg::dedup_scatter_kernel<<<blocks, 256, 0, st>>>(d_si, d_scan, d_pos, n, d_rf);   // d_rf is free after the run sort
        g_launches++;
        if (read_to_distinct) CU_TRY(cudaMemcpyAsync(read_to_distinct, d_rf, R * 4, cudaMemcpyDeviceToHost, st));
    }
    CU_TRY(cudaGetLastError());
    CU_TRY(cudaStreamSynchronize(st));
    *n_distinct = n_runs;
    return BDG_OK;
}

int bdg_dedup_first_seen(const uint32_t* ranks, size_t R, uint32_t* distinct, uint32_t* counts, uint32_t* read_to_distinct,
                         uint32_t* sorted_pos, size_t* n_distinct)
{
    if (!n_distinct) return fail(BDG_ERR_ARG, "NULL n_distinct pointer");
    *n_distinct = 0;
    if (R == 0) return BDG_OK;
    if (!ranks || !distinct || !counts) return fail(BDG_ERR_ARG, "NULL pointer argument");
    if (R > 0x7FFFFFFFull) return fail(BDG_ERR_ARG, "more than 2^31 reads in one call");
    if (int rc = need_ctx()) return rc;
    DevCtx& c = g_ctx[0];
    CU_TRY(cudaSetDevice(c.dev));
    c.map.drop();
    if (int e = c.map.keys().ensure(R * 4)) return e;
    CU_TRY(cudaMemcpyAsync(c.map.keys().p, ranks, R * 4, cudaMemcpyHostToDevice, c.stream));
    return dedup_core(c, (uint32_t)R, distinct, counts, read_to_distinct, sorted_pos, false, n_distinct);
}

// ---- f-1 + f-2 on the device: masked dedup that keeps the read map resident, and the per-read gather that uses it ------
// ranks / valid are host arrays (kind = cudaMemcpyHostToDevice) or device arrays on c.dev (cudaMemcpyDeviceToDevice): the masked
// compaction reads device ranks in place (host ranks are uploaded into c.io first); the valid bytes are always copied, because
// the per-read gather reads them again.
static int dedup_reads_core(DevCtx& c, const uint32_t* ranks, const uint8_t* valid, size_t R_all, cudaMemcpyKind kind, uint32_t* distinct,
                            uint32_t* counts, uint32_t* sorted_pos, uint32_t* sorted_distinct, size_t* n_distinct, size_t* n_valid,
                            unsigned long long* token)
{
    cudaStream_t st = c.stream;
    ReadMap& m = c.map;
    m.drop();
    if (int e = m.keys().ensure(R_all * 4)) return e;
    size_t n_reads = R_all;
    m.masked = valid != nullptr;
    if (valid) {
        // the valid bytes and their scan stay with the read map
        if (int e = m.valid.ensure(R_all)) return e;
        if (int e = m.valid_scan.ensure((R_all + 1) * 4)) return e;
        const uint8_t* d_valid = (const uint8_t*)m.valid.p;
        uint32_t* d_excl = (uint32_t*)m.valid_scan.p;
        auto flags = thrust::make_transform_iterator(d_valid, bdg::NonZero());
        size_t tmp = 0;
        CU_TRY(cub::DeviceScan::ExclusiveSum(nullptr, tmp, flags, d_excl, (int)R_all, st));
        if (int e = c.mask_tmp.ensure(tmp)) return e;
        const uint32_t* d_ranks = ranks;
        if (kind == cudaMemcpyHostToDevice) {
            uint32_t* up = nullptr;
            if (int e = stage(c, {piece(up, R_all * 4)})) return e;
            CU_TRY(cudaMemcpyAsync(up, ranks, R_all * 4, kind, st));
            d_ranks = up;
        }
        CU_TRY(cudaMemcpyAsync(m.valid.p, valid, R_all, kind, st));
        CU_TRY(cub::DeviceScan::ExclusiveSum(c.mask_tmp.p, tmp, flags, d_excl, (int)R_all, st));
        const int blocks = (int)std::min<size_t>((R_all + 255) / 256, (size_t)c.sms * 8);
        bdg::compact_valid_kernel<<<blocks, 256, 0, st>>>(d_ranks, d_valid, d_excl, (uint32_t)R_all, (uint32_t*)m.keys().p);
        g_launches++;
        uint32_t last_excl = 0;
        uint8_t last_valid = 0;
        CU_TRY(cudaMemcpyAsync(&last_excl, d_excl + (R_all - 1), 4, cudaMemcpyDeviceToHost, st));
        CU_TRY(cudaMemcpyAsync(&last_valid, d_valid + (R_all - 1), 1, cudaMemcpyDeviceToHost, st));
        CU_TRY(cudaStreamSynchronize(st));
        n_reads = (size_t)last_excl + (last_valid ? 1 : 0);
    } else {
        CU_TRY(cudaMemcpyAsync(m.keys().p, ranks, R_all * 4, kind, st));
    }
    *n_valid = n_reads;
    m.rows = R_all; m.reads = n_reads; m.distinct = 0;
    if (n_reads == 0) return BDG_OK;
    if (int rc = dedup_core(c, (uint32_t)n_reads, distinct, counts, nullptr, sorted_pos, true, n_distinct, sorted_distinct)) return rc;
    return m.install(*n_distinct, nullptr, nullptr, nullptr, nullptr, st, token);       // dedup_core left the arrays in place
}

static int dedup_reads_args(const uint32_t* ranks, size_t R_all, size_t* n_distinct, size_t* n_valid, unsigned long long* token, DevCtx** c)
{
    if (!n_distinct || !n_valid || !token) return fail(BDG_ERR_ARG, "NULL result pointer");
    *n_distinct = 0; *n_valid = 0; *token = 0;
    if (R_all == 0) return EMPTY;
    if (!ranks) return fail(BDG_ERR_ARG, "NULL pointer argument");
    if (R_all > 0x7FFFFFFFull) return fail(BDG_ERR_ARG, "more than 2^31 reads in one call");
    return first_ctx(c);
}

// The host form downloads the outputs it was given (kind = cudaMemcpyHostToDevice; see dedup_reads_core), the device form has none.
static int dedup_reads_body(DevCtx& c, const uint32_t* ranks, const uint8_t* valid, size_t R_all, cudaMemcpyKind kind, uint32_t* distinct,
                            uint32_t* counts, uint32_t* sorted_pos, uint32_t* sorted_distinct, size_t* n_distinct, size_t* n_valid,
                            unsigned long long* token, cudaStream_t caller)
{
    CallerOrder order(c, caller);
    if (int rc = order.begin()) return rc;
    return dedup_reads_core(c, ranks, valid, R_all, kind, distinct, counts, sorted_pos, sorted_distinct, n_distinct, n_valid, token);
}

int bdg_dedup_reads(const uint32_t* ranks, const uint8_t* valid, size_t R_all, uint32_t* distinct, uint32_t* counts, uint32_t* sorted_pos,
                    uint32_t* sorted_distinct, size_t* n_distinct, size_t* n_valid, unsigned long long* token)
{
    DevCtx* c = nullptr;
    if (int rc = dedup_reads_args(ranks, R_all, n_distinct, n_valid, token, &c)) return done(rc);
    return dedup_reads_body(*c, ranks, valid, R_all, cudaMemcpyHostToDevice, distinct, counts, sorted_pos, sorted_distinct, n_distinct, n_valid,
                            token, c->stream);
}

int bdg_dev_dedup_reads(const uint32_t* d_ranks, const uint8_t* d_valid, size_t R_all, size_t* n_distinct, size_t* n_valid,
                        unsigned long long* token, void* stream)
{
    DevCtx* c = nullptr;
    if (int rc = dedup_reads_args(d_ranks, R_all, n_distinct, n_valid, token, &c)) return done(rc);
    if (int rc = check_on_first(d_ranks, "ranks")) return rc;
    if (d_valid) if (int rc = check_on_first(d_valid, "valid")) return rc;
    return dedup_reads_body(*c, d_ranks, d_valid, R_all, cudaMemcpyDeviceToDevice, nullptr, nullptr, nullptr, nullptr, n_distinct, n_valid, token,
                            (cudaStream_t)stream);
}

// What bdg_dedup_reads left on the device, on demand (any pointer may be NULL): the arrays of its output list, to the host
// (kind = cudaMemcpyDeviceToHost, the call waits for the copies) or to device memory on c.dev (stream-ordered, no wait).
static int dedup_fetch_body(DevCtx& c, uint32_t* distinct, uint32_t* counts, uint32_t* sorted_pos, uint32_t* sorted_distinct, cudaMemcpyKind kind,
                            cudaStream_t caller)
{
    CallerOrder order(c, caller);
    if (int rc = order.begin()) return rc;
    const ReadMap& m = c.map;
    const size_t n = m.distinct;
    if (distinct) CU_TRY(cudaMemcpyAsync(distinct, m.first_seen(), n * 4, kind, c.stream));
    if (counts) CU_TRY(cudaMemcpyAsync(counts, m.counts(), n * 4, kind, c.stream));
    if (sorted_pos) CU_TRY(cudaMemcpyAsync(sorted_pos, m.order(), n * 4, kind, c.stream));
    if (sorted_distinct) CU_TRY(cudaMemcpyAsync(sorted_distinct, m.ascending(), n * 4, kind, c.stream));
    if (kind == cudaMemcpyDeviceToHost) CU_TRY(cudaStreamSynchronize(c.stream));
    return BDG_OK;
}

int bdg_dedup_fetch(unsigned long long token, uint32_t* distinct, uint32_t* counts, uint32_t* sorted_pos, uint32_t* sorted_distinct)
{
    DevCtx* c = nullptr;
    if (int rc = map_ctx(token, &c)) return rc;
    return dedup_fetch_body(*c, distinct, counts, sorted_pos, sorted_distinct, cudaMemcpyDeviceToHost, c->stream);
}

int bdg_dev_dedup_fetch(unsigned long long token, uint32_t* d_distinct, uint32_t* d_counts, uint32_t* d_sorted_pos, uint32_t* d_sorted_distinct,
                        void* stream)
{
    DevCtx* c = nullptr;
    if (int rc = map_ctx(token, &c)) return rc;
    for (uint32_t* p : {d_distinct, d_counts, d_sorted_pos, d_sorted_distinct})
        if (p && c->map.distinct) if (int rc = check_on_first(p, "output")) return rc;
    return dedup_fetch_body(*c, d_distinct, d_counts, d_sorted_pos, d_sorted_distinct, cudaMemcpyDeviceToDevice, (cudaStream_t)stream);
}

// ---- the dedup results of P parts (one process per GPU) reduced to the global distinct set (bdg_kernels.cuh, merge_*) ----
// The work arrays live in c.mg until the end, so that a failed check leaves the token's read map as it was; only then are the
// global arrays installed as the read map (counts, order, first-seen, ascending) and its read_pos rewritten in place.  The valid
// rows are not touched.
static int dedup_merge_core(DevCtx& c, const uint32_t* d_keys, const uint32_t* d_counts, const uint32_t* d_first, const size_t* starts,
                            const size_t* sizes, int n_parts, int my_part, size_t* n_distinct, unsigned long long* merged_token)
{
    cudaStream_t st = c.stream;
    std::vector<uint64_t> h_starts(n_parts);
    std::vector<uint32_t> h_offs(n_parts + 1, 0);
    size_t total = 0;
    for (int p = 0; p < n_parts; p++) {
        h_starts[p] = starts[p];
        h_offs[p] = (uint32_t)total;
        total += sizes[p];
        if (total >= 0x80000000ull) return fail(BDG_ERR_ARG, "the parts hold 2^31 or more barcodes in all");
    }
    h_offs[n_parts] = (uint32_t)total;
    if (total == 0) return fail(BDG_ERR_ARG, "no part holds a barcode");
    const uint32_t T = (uint32_t)total, n_mine = (uint32_t)sizes[my_part], off_mine = h_offs[my_part];
    // mg.head also holds the run order, mg.scan the sorted first keys; mg.runs: run key | count | first | own run | position of run | local -> global
    auto& g = c.mg;
    if (int e = g.starts.ensure((size_t)n_parts * 8)) return e;
    if (int e = g.offs.ensure(((size_t)n_parts + 1) * 4 + 4)) return e;
    for (Buf* b : {&g.key, &g.idx, &g.sorted_key, &g.sorted_idx, &g.cnt, &g.first, &g.head, &g.scan}) if (int e = b->ensure(total * 4)) return e;
    if (int e = g.runs.ensure((5 * total + std::max<size_t>(n_mine, 1)) * 4)) return e;
    uint32_t *d_key = (uint32_t*)g.key.p, *d_idx = (uint32_t*)g.idx.p, *d_sk = (uint32_t*)g.sorted_key.p, *d_si = (uint32_t*)g.sorted_idx.p;
    uint32_t *d_cnt = (uint32_t*)g.cnt.p, *d_fst = (uint32_t*)g.first.p, *d_head = (uint32_t*)g.head.p, *d_scan = (uint32_t*)g.scan.p;
    uint32_t *d_rk = (uint32_t*)g.runs.p, *d_rc = d_rk + total, *d_rf = d_rc + total, *d_mrun = d_rf + total, *d_prun = d_mrun + total,
             *d_loc = d_prun + total;
    unsigned int* d_bad = (unsigned int*)((uint32_t*)g.offs.p + n_parts + 1);
    size_t tmp1 = 0, tmp2 = 0;
    CU_TRY(cub::DeviceRadixSort::SortPairs(nullptr, tmp1, d_key, d_sk, d_idx, d_si, (int)T, 0, 32, st));
    CU_TRY(cub::DeviceScan::InclusiveSum(nullptr, tmp2, d_head, d_scan, (int)T, st));
    if (int e = g.tmp.ensure(std::max(tmp1, tmp2))) return e;
    CU_TRY(cudaMemcpyAsync(g.starts.p, h_starts.data(), (size_t)n_parts * 8, cudaMemcpyHostToDevice, st));
    CU_TRY(cudaMemcpyAsync(g.offs.p, h_offs.data(), ((size_t)n_parts + 1) * 4, cudaMemcpyHostToDevice, st));
    CU_TRY(cudaMemsetAsync(d_bad, 0, 4, st));
    const int blocks = (int)std::min<size_t>((total + 255) / 256, (size_t)c.sms * 8);
    bdg::merge_gather_kernel<<<blocks, 256, 0, st>>>(d_keys, d_counts, d_first, (const uint64_t*)g.starts.p, (const uint32_t*)g.offs.p, (uint32_t)n_parts,
                                                     T, (uint32_t)my_part, c.map.ascending(), d_key, d_idx, d_cnt, d_fst, d_bad);
    CU_TRY(cub::DeviceRadixSort::SortPairs(g.tmp.p, tmp1, d_key, d_sk, d_idx, d_si, (int)T, 0, 32, st));
    bdg::dedup_heads_kernel<<<blocks, 256, 0, st>>>(d_sk, T, d_head);
    CU_TRY(cub::DeviceScan::InclusiveSum(g.tmp.p, tmp2, d_head, d_scan, (int)T, st));
    bdg::merge_runs_kernel<<<blocks, 256, 0, st>>>(d_sk, d_si, d_head, d_scan, T, d_cnt, d_fst, off_mine, n_mine, d_rk, d_rc, d_rf, d_mrun);
    g_launches += 3;
    CU_TRY(cudaGetLastError());
    uint32_t n_runs = 0;
    unsigned int bad = 0;
    CU_TRY(cudaMemcpyAsync(&n_runs, d_scan + (T - 1), 4, cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaMemcpyAsync(&bad, d_bad, 4, cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaStreamSynchronize(st));
    if (bad) return fail(BDG_ERR_ARG, "the list of part %d is not the distinct list of the read map the token names", my_part);
    // runs by first key (unique: every key names one barcode of one part): d_scan := sorted first keys, d_head := order
    bdg::iota_kernel<<<blocks, 256, 0, st>>>(d_idx, n_runs);
    CU_TRY(cub::DeviceRadixSort::SortPairs(g.tmp.p, tmp1, d_rf, d_scan, d_idx, d_head, (int)n_runs, 0, 32, st));
    // d_key / d_cnt are free: distinct and counts in first-seen order
    bdg::merge_finish_kernel<<<blocks, 256, 0, st>>>(d_head, d_rk, d_rc, n_runs, d_key, d_cnt, d_prun);
    g_launches += 2;
    if (n_mine) {
        const int lb = (int)std::min<size_t>((n_mine + 255) / 256, (size_t)c.sms * 8);
        const int rb = (int)std::min<size_t>((c.map.reads + 255) / 256, (size_t)c.sms * 8);
        bdg::merge_local_kernel<<<lb, 256, 0, st>>>(c.map.order(), d_mrun, d_prun, n_mine, d_loc);
        bdg::merge_remap_kernel<<<rb, 256, 0, st>>>(c.map.read_pos(), (uint32_t)c.map.reads, d_loc);
        g_launches += 2;
    }
    CU_TRY(cudaGetLastError());
    // order[pos] = run = ascending position; runs are numbered in key order
    if (int rc = c.map.install(n_runs, d_cnt, d_head, d_key, d_rk, st, merged_token)) return rc;
    *n_distinct = n_runs;
    return BDG_OK;
}

int bdg_dev_dedup_merge(unsigned long long token, const uint32_t* d_keys, const uint32_t* d_counts, const uint32_t* d_first, const size_t* starts,
                        const size_t* sizes, int n_parts, int my_part, size_t* n_distinct, unsigned long long* merged_token, void* stream)
{
    if (!n_distinct || !merged_token) return fail(BDG_ERR_ARG, "NULL result pointer");
    *n_distinct = 0; *merged_token = 0;
    if (n_parts < 1 || my_part < 0 || my_part >= n_parts || !starts || !sizes) return fail(BDG_ERR_ARG, "need 0 <= my_part < n_parts and the parts' starts / sizes");
    if (!d_keys || !d_counts || !d_first) return fail(BDG_ERR_ARG, "NULL pointer argument");
    // token 0: this part has no valid read (the dedup call issued no token); its list must then be empty
    DevCtx* cp = nullptr;
    if (token != 0) {
        if (int rc = map_ctx(token, &cp)) return rc;
    } else {
        if (int rc = need_ctx()) return rc;
        cp = &g_ctx[0];
        CU_TRY(cudaSetDevice(cp->dev));
    }
    DevCtx& c = *cp;
    if (sizes[my_part] != (token ? c.map.distinct : 0))
        return fail(BDG_ERR_ARG, "part %d has %zu barcodes, the read map of the token %zu", my_part, sizes[my_part], token ? c.map.distinct : (size_t)0);
    for (const uint32_t* p : {d_keys, d_counts, d_first}) if (int rc = check_on_first(p, "merge input")) return rc;
    if (token == 0) { c.map.drop(); c.map.rows = 0; c.map.reads = 0; c.map.masked = false; }
    CallerOrder order(c, stream);
    if (int rc = order.begin()) return rc;
    return dedup_merge_core(c, d_keys, d_counts, d_first, starts, sizes, n_parts, my_part, n_distinct, merged_token);
}

}  // extern "C"

// ---- the tally: reads deduplicated batch by batch into a running distinct set (bdg_kernels.cuh, tally_*) -------------------
// The set lives in the handle's own buffers, ascending by barcode, with a 64-bit count and a 64-bit first-sighting key per
// barcode: the rows added before the batch + the barcode's first-seen position in the batch, so that the keys sort in the
// first-seen order of the concatenated batches.  add merges a batch into the other half of the double buffer and swaps; a
// refused batch leaves the set as it was.  finish sorts the set by first-sighting key and installs the read-map arrays of a
// dedup call without rows (counts, first-seen -> ascending, distinct in first-seen order, ascending).
struct bdg_tally {
    int dev = -1;                                   // the first claimed device when the tally was created
    Buf key[2], cnt[2], fst[2];                     // the running set and the half the next batch is merged into
    Buf m_key, m_cnt, m_fst, m_head, m_scan;        // the merged order of set and batch, head flags and their scan; order at finish
    Buf scratch, flag;                              // cub scratch; overflow flag + set size read back after a merge
    int cur = 0;
    size_t n = 0;                                   // distinct barcodes in the set
    unsigned long long rows = 0, valid = 0;         // rows and valid rows added
    bool over = false;                              // some barcode was counted 2^32 times or more
    bool finished = false;
};

namespace {

int tally_ready(bdg_tally* h, DevCtx** out)
{
    if (!h) return fail(BDG_ERR_ARG, "NULL tally handle");
    if (g_ctx.empty() || g_ctx[0].dev != h->dev)
        return fail(BDG_ERR_ARG, "the tally lives on device %d, which is not the first claimed device", h->dev);
    *out = &g_ctx[0];
    CU_TRY(cudaSetDevice(h->dev));
    return BDG_OK;
}

// One merge of the B side into the set of src_n entries in key[src] (merge path, scan of the heads, compaction into key[dst]):
// *n_out = entries of the new set, *over = some count reached 2^32.  Waits for both.
template <typename BSide>
int tally_merge_step(DevCtx& c, bdg_tally* h, int src, size_t src_n, int dst, const BSide& b, uint32_t* n_out, bool* over)
{
    cudaStream_t st = c.stream;
    const size_t na = src_n, M = na + b.n;          // na < 2^31 and nb < 2^31: M < 2^32
    for (Buf* x : {&h->m_key, &h->m_head, &h->m_scan, &h->key[dst]}) if (int e = x->ensure(M * 4)) return e;
    for (Buf* x : {&h->m_cnt, &h->m_fst, &h->cnt[dst], &h->fst[dst]}) if (int e = x->ensure(M * 8)) return e;
    if (int e = h->flag.ensure(16)) return e;
    size_t tmp = 0;
    CU_TRY(cub::DeviceScan::InclusiveSum(nullptr, tmp, (const uint32_t*)h->m_head.p, (uint32_t*)h->m_scan.p, (int64_t)M, st));
    if (int e = h->scratch.ensure(tmp)) return e;
    unsigned int* d_flag = (unsigned int*)h->flag.p;
    CU_TRY(cudaMemsetAsync(d_flag, 0, 4, st));
    bdg::tally_merge_kernel<BSide><<<(unsigned)((M + bdg::TALLY_TILE - 1) / bdg::TALLY_TILE), bdg::NT, 0, st>>>(
        (const uint32_t*)h->key[src].p, (const unsigned long long*)h->cnt[src].p, (const unsigned long long*)h->fst[src].p, na, b.key, b.x,
        b.y, b.n, b.first_off, (uint32_t*)h->m_key.p, (unsigned long long*)h->m_cnt.p, (unsigned long long*)h->m_fst.p, (uint32_t*)h->m_head.p);
    CU_TRY(cub::DeviceScan::InclusiveSum(h->scratch.p, tmp, (const uint32_t*)h->m_head.p, (uint32_t*)h->m_scan.p, (int64_t)M, st));
    const int blocks = (int)std::min<size_t>((M + 255) / 256, (size_t)c.sms * 8);
    bdg::tally_compact_kernel<<<blocks, 256, 0, st>>>((const uint32_t*)h->m_key.p, (const unsigned long long*)h->m_cnt.p,
                                                      (const unsigned long long*)h->m_fst.p, (const uint32_t*)h->m_head.p,
                                                      (const uint32_t*)h->m_scan.p, M, (uint32_t*)h->key[dst].p,
                                                      (unsigned long long*)h->cnt[dst].p, (unsigned long long*)h->fst[dst].p, d_flag);
    g_launches += 2;
    CU_TRY(cudaGetLastError());
    uint32_t over_flag = 0;
    CU_TRY(cudaMemcpyAsync(n_out, (const uint32_t*)h->m_scan.p + (M - 1), 4, cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaMemcpyAsync(&over_flag, d_flag, 4, cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaStreamSynchronize(st));
    *over = over_flag != 0;
    return BDG_OK;
}

int tally_add_args(bdg_tally* h, const uint32_t* ranks, size_t R, size_t* n_valid, DevCtx** c)
{
    if (n_valid) *n_valid = 0;
    if (int rc = tally_ready(h, c)) return rc;
    if (h->finished) return fail(BDG_ERR_ARG, "add after finish: the tally is closed");
    if (R == 0) return EMPTY;
    if (!ranks) return fail(BDG_ERR_ARG, "NULL pointer argument");
    if (R > 0x7FFFFFFFull) return fail(BDG_ERR_ARG, "more than 2^31 reads in one call");
    return BDG_OK;
}

// ranks / valid as for dedup_reads_core
int tally_add_body(DevCtx& c, bdg_tally* h, const uint32_t* ranks, const uint8_t* valid, size_t R, cudaMemcpyKind kind, size_t* n_valid,
                   cudaStream_t caller)
{
    CallerOrder order(c, caller);
    if (int rc = order.begin()) return rc;
    size_t nb = 0, nv = 0;
    unsigned long long tok = 0;
    const int rc = dedup_reads_core(c, ranks, valid, R, kind, nullptr, nullptr, nullptr, nullptr, &nb, &nv, &tok);
    c.map.drop();                                   // the batch's read map is not handed out
    if (rc) return rc;
    if (n_valid) *n_valid = nv;
    if (nv == 0) { h->rows += R; return BDG_OK; }
    const int nx = h->cur ^ 1;
    const bdg::TallyBatchSide batch{c.map.ascending() /* batch runs ascending */, c.map.counts() /* counts, first-seen order */,
                                    c.map.run_pos() /* run -> first-seen position */, nb, h->rows};
    uint32_t n_out = 0;
    bool over = false;
    if (int e = tally_merge_step(c, h, h->cur, h->n, nx, batch, &n_out, &over)) return e;
    if (n_out > 0x7FFFFFFFu)
        return fail(BDG_ERR_ARG, "the batch would take the tally to %u distinct barcodes; fewer than 2^31 are allowed (the set keeps the batches before it)", n_out);
    h->cur = nx;
    h->n = n_out;
    h->rows += R;
    h->valid += nv;
    h->over = h->over || over;
    return BDG_OK;
}

// The P parts' sets folded into one, part 0 first: every step merges the next part into the running union, alternating between the
// handle's two halves.  The checks run first; a refusal after the fold began restores the handle's set from the caller's own
// part, which the checks found equal to it entry for entry.
int tally_merge_parts_core(DevCtx& c, bdg_tally* h, const uint32_t* d_keys, const unsigned long long* d_cnts, const unsigned long long* d_firsts,
                           const size_t* starts, const size_t* sizes, const unsigned long long* row_offsets, int n_parts, int my_part,
                           unsigned long long total_rows, unsigned long long total_valid)
{
    cudaStream_t st = c.stream;
    auto part = [&](int p) {
        return bdg::TallySetSide{d_keys + starts[p], d_cnts + starts[p], d_firsts + starts[p], (uint64_t)sizes[p], row_offsets[p]};
    };
    if (int e = h->flag.ensure(16)) return e;
    unsigned int* d_flag = (unsigned int*)h->flag.p;
    CU_TRY(cudaMemsetAsync(d_flag, 0, 4, st));
    for (int p = 0; p < n_parts; p++) {
        if (!sizes[p]) continue;
        const bool mine = p == my_part;
        const int blocks = (int)std::min<size_t>((sizes[p] + 255) / 256, (size_t)c.sms * 8);
        bdg::tally_part_check_kernel<<<blocks, 256, 0, st>>>(part(p), total_rows, mine ? (const uint32_t*)h->key[h->cur].p : nullptr,
                                                             mine ? (const unsigned long long*)h->cnt[h->cur].p : nullptr,
                                                             mine ? (const unsigned long long*)h->fst[h->cur].p : nullptr, d_flag);
        g_launches++;
    }
    CU_TRY(cudaGetLastError());
    unsigned int bad = 0;
    CU_TRY(cudaMemcpyAsync(&bad, d_flag, 4, cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaStreamSynchronize(st));
    if (bad & 1u) return fail(BDG_ERR_ARG, "the barcodes of a part are not strictly ascending");
    if (bad & 2u) return fail(BDG_ERR_ARG, "part %d is not the tally's own set", my_part);
    if (bad & 4u) return fail(BDG_ERR_ARG, "a shifted first sighting is not below the %llu rows of all parts", total_rows);

    auto restore = [&]() {
        const size_t n = h->n, s = starts[my_part];   // key[cur] still has room for n entries: buffers only grow
        if (n == 0) return;
        cudaMemcpyAsync(h->key[h->cur].p, d_keys + s, n * 4, cudaMemcpyDeviceToDevice, st);
        cudaMemcpyAsync(h->cnt[h->cur].p, d_cnts + s, n * 8, cudaMemcpyDeviceToDevice, st);
        cudaMemcpyAsync(h->fst[h->cur].p, d_firsts + s, n * 8, cudaMemcpyDeviceToDevice, st);
        cudaStreamSynchronize(st);
    };
    int cur = h->cur;
    size_t n = 0;
    bool over = false;
    for (int p = 0; p < n_parts; p++) {
        if (!sizes[p]) continue;
        uint32_t n_out = 0;
        bool o = false;
        if (int e = tally_merge_step(c, h, cur, n, cur ^ 1, part(p), &n_out, &o)) {
            restore();
            return e;
        }
        if (n_out > 0x7FFFFFFFu) {
            restore();
            return fail(BDG_ERR_ARG, "the parts hold %u or more distinct barcodes in all; fewer than 2^31 are allowed", n_out);
        }
        cur ^= 1;
        n = n_out;
        over = over || o;
    }
    h->cur = cur;
    h->n = n;
    h->rows = total_rows;
    h->valid = total_valid;
    h->over = over;                                 // from the merged counts alone: the same on every part
    h->finished = true;                             // the set holds the other parts' batches: no batch can follow them
    return BDG_OK;
}

int tally_finish_args(bdg_tally* h, size_t* n_distinct, size_t* n_valid, unsigned long long* token, DevCtx** c)
{
    if (!n_distinct || !n_valid || !token) return fail(BDG_ERR_ARG, "NULL result pointer");
    *n_distinct = 0; *n_valid = 0; *token = 0;
    return tally_ready(h, c);
}

int tally_finish_body(DevCtx& c, bdg_tally* h, size_t* n_distinct, size_t* n_valid, unsigned long long* token, cudaStream_t caller)
{
    CallerOrder order(c, caller);
    if (int rc = order.begin()) return rc;
    if (h->over) return fail(BDG_ERR_ARG, "a barcode was counted 2^32 times or more; the counts of a read map are uint32");
    *n_valid = h->valid;
    h->finished = true;
    if (h->n == 0) return BDG_OK;                   // no valid row: no read map, as with a dedup call
    cudaStream_t st = c.stream;
    const uint32_t n = (uint32_t)h->n;
    int end_bit = 1;                                // every first-sighting key is below the number of rows added
    while (end_bit < 64 && (h->rows >> end_bit)) end_bit++;
    // m_key := iota, m_fst := sorted keys, m_head := order (all hold >= n entries since the merge that made the set)
    size_t tmp = 0;
    CU_TRY(cub::DeviceRadixSort::SortPairs(nullptr, tmp, (const unsigned long long*)h->fst[h->cur].p, (unsigned long long*)h->m_fst.p,
                                           (const uint32_t*)h->m_key.p, (uint32_t*)h->m_head.p, (int)n, 0, end_bit, st));
    if (int e = h->scratch.ensure(tmp)) return e;
    const int blocks = (int)std::min<size_t>((n + 255) / 256, (size_t)c.sms * 8);
    bdg::iota_kernel<<<blocks, 256, 0, st>>>((uint32_t*)h->m_key.p, n);
    CU_TRY(cub::DeviceRadixSort::SortPairs(h->scratch.p, tmp, (const unsigned long long*)h->fst[h->cur].p, (unsigned long long*)h->m_fst.p,
                                           (const uint32_t*)h->m_key.p, (uint32_t*)h->m_head.p, (int)n, 0, end_bit, st));
    g_launches++;
    // the ascending array is the set itself; first-seen, counts and order are written in place by the kernel below
    c.map.rows = 0; c.map.reads = 0; c.map.masked = false;
    unsigned long long tok = 0;
    if (int rc = c.map.install(n, nullptr, nullptr, nullptr, (const uint32_t*)h->key[h->cur].p, st, &tok)) return rc;
    bdg::tally_finish_kernel<<<blocks, 256, 0, st>>>((const uint32_t*)h->m_head.p, (const uint32_t*)h->key[h->cur].p,
                                                     (const unsigned long long*)h->cnt[h->cur].p, n, c.map.first_seen(), c.map.counts(),
                                                     c.map.order());
    g_launches++;
    if (cudaError_t e = cudaGetLastError()) {
        c.map.drop();
        return fail(BDG_ERR_CUDA, "tally finish launch failed: %s", cudaGetErrorString(e));
    }
    *n_distinct = n;
    *token = tok;
    return BDG_OK;
}

}  // namespace

extern "C" {

int bdg_tally_create(bdg_tally** out)
{
    if (!out) return fail(BDG_ERR_ARG, "NULL pointer argument");
    *out = nullptr;
    if (int rc = need_ctx()) return rc;
    bdg_tally* h = new (std::nothrow) bdg_tally();
    if (!h) return fail(BDG_ERR_OOM, "host allocation failed");
    h->dev = g_ctx[0].dev;
    *out = h;
    return BDG_OK;
}

void bdg_tally_free(bdg_tally* h)
{
    if (!h) return;
    int prev = -1;
    cudaGetDevice(&prev);
    cudaSetDevice(h->dev);                          // the buffers are freed on their device
    delete h;
    if (prev >= 0) cudaSetDevice(prev);
}

int bdg_tally_add(bdg_tally* h, const uint32_t* ranks, const uint8_t* valid, size_t R, size_t* n_valid)
{
    DevCtx* c = nullptr;
    if (int rc = tally_add_args(h, ranks, R, n_valid, &c)) return done(rc);
    return tally_add_body(*c, h, ranks, valid, R, cudaMemcpyHostToDevice, n_valid, c->stream);
}

int bdg_dev_tally_add(bdg_tally* h, const uint32_t* d_ranks, const uint8_t* d_valid, size_t R, size_t* n_valid, void* stream)
{
    DevCtx* c = nullptr;
    if (int rc = tally_add_args(h, d_ranks, R, n_valid, &c)) return done(rc);
    if (int rc = check_on_first(d_ranks, "ranks")) return rc;
    if (d_valid) if (int rc = check_on_first(d_valid, "valid")) return rc;
    return tally_add_body(*c, h, d_ranks, d_valid, R, cudaMemcpyDeviceToDevice, n_valid, (cudaStream_t)stream);
}

int bdg_tally_finish(bdg_tally* h, size_t* n_distinct, size_t* n_valid, unsigned long long* token)
{
    DevCtx* c = nullptr;
    if (int rc = tally_finish_args(h, n_distinct, n_valid, token, &c)) return rc;
    return tally_finish_body(*c, h, n_distinct, n_valid, token, c->stream);
}

int bdg_dev_tally_finish(bdg_tally* h, size_t* n_distinct, size_t* n_valid, unsigned long long* token, void* stream)
{
    DevCtx* c = nullptr;
    if (int rc = tally_finish_args(h, n_distinct, n_valid, token, &c)) return rc;
    return tally_finish_body(*c, h, n_distinct, n_valid, token, (cudaStream_t)stream);
}

int bdg_tally_info(bdg_tally* h, size_t* n_distinct, unsigned long long* rows, unsigned long long* valid)
{
    if (!n_distinct || !rows || !valid) return fail(BDG_ERR_ARG, "NULL result pointer");
    *n_distinct = 0; *rows = 0; *valid = 0;
    DevCtx* c = nullptr;
    if (int rc = tally_ready(h, &c)) return rc;
    *n_distinct = h->n;
    *rows = h->rows;
    *valid = h->valid;
    return BDG_OK;
}

int bdg_dev_tally_copy(bdg_tally* h, uint32_t* d_key, unsigned long long* d_cnt, unsigned long long* d_first, void* stream)
{
    DevCtx* c = nullptr;
    if (int rc = tally_ready(h, &c)) return rc;
    if (h->n == 0) return BDG_OK;
    if (!d_key || !d_cnt || !d_first) return fail(BDG_ERR_ARG, "NULL pointer argument");
    for (const void* p : {(const void*)d_key, (const void*)d_cnt, (const void*)d_first})
        if (int rc = check_on_first(p, "output")) return rc;
    CallerOrder order(*c, stream);
    if (int rc = order.begin()) return rc;
    cudaStream_t st = c->stream;
    CU_TRY(cudaMemcpyAsync(d_key, h->key[h->cur].p, h->n * 4, cudaMemcpyDeviceToDevice, st));
    CU_TRY(cudaMemcpyAsync(d_cnt, h->cnt[h->cur].p, h->n * 8, cudaMemcpyDeviceToDevice, st));
    CU_TRY(cudaMemcpyAsync(d_first, h->fst[h->cur].p, h->n * 8, cudaMemcpyDeviceToDevice, st));
    return BDG_OK;
}

int bdg_dev_tally_merge_parts(bdg_tally* h, const uint32_t* d_keys, const unsigned long long* d_cnts, const unsigned long long* d_firsts,
                              const size_t* starts, const size_t* sizes, const unsigned long long* row_offsets, int n_parts, int my_part,
                              unsigned long long total_rows, unsigned long long total_valid, void* stream)
{
    DevCtx* c = nullptr;
    if (int rc = tally_ready(h, &c)) return rc;
    if (h->finished) return fail(BDG_ERR_ARG, "merge after finish: the tally is closed");
    if (n_parts < 1 || my_part < 0 || my_part >= n_parts || !starts || !sizes || !row_offsets)
        return fail(BDG_ERR_ARG, "need 0 <= my_part < n_parts and the parts' starts / sizes / row offsets");
    if (sizes[my_part] != h->n) return fail(BDG_ERR_ARG, "part %d has %zu barcodes, the tally's set %zu", my_part, sizes[my_part], h->n);
    if (total_rows < h->rows || total_valid < h->valid || total_valid > total_rows)
        return fail(BDG_ERR_ARG, "%llu rows / %llu valid rows in all, but the tally alone added %llu / %llu", total_rows, total_valid,
                    h->rows, h->valid);
    size_t total = 0;
    for (int p = 0; p < n_parts; p++) {
        if (sizes[p] > 0x7FFFFFFFull) return fail(BDG_ERR_ARG, "part %d has %zu barcodes; fewer than 2^31 are allowed", p, sizes[p]);
        total += sizes[p];
    }
    if (total) {
        if (!d_keys || !d_cnts || !d_firsts) return fail(BDG_ERR_ARG, "NULL pointer argument");
        for (const void* p : {(const void*)d_keys, (const void*)d_cnts, (const void*)d_firsts})
            if (int rc = check_on_first(p, "merge input")) return rc;
    }
    CallerOrder order(*c, stream);
    if (int rc = order.begin()) return rc;
    return tally_merge_parts_core(*c, h, d_keys, d_cnts, d_firsts, starts, sizes, row_offsets, n_parts, my_part, total_rows, total_valid);
}

// ---- a-6 / centre selection, barcode_graph.py:252-267, over the distinct barcodes a dedup call left on the device ----
// cutoff = max(mean(counts of the first n_cells barcodes in first-seen order) / 5, 5) (:255-256); the barcodes with
// count > cutoff in count-descending order, ties in first-seen order (the head of `bc_by_counts`, :253), with their counts and
// - when a whitelist is given - their membership (:264).  The short walk over that head stays with the caller.
// sorted_wl is a host array (wl_on_device false: uploaded into c.io) or device memory on c.dev, read in place.
static int centres_above_body(DevCtx& c, size_t n_cells, const uint32_t* sorted_wl, bool wl_on_device, size_t W, uint32_t* top_ranks,
                              uint32_t* top_counts, uint8_t* top_hits, size_t cap, size_t* n_above, double* cutoff, cudaStream_t caller)
{
    CallerOrder order(c, caller);
    if (int rc = order.begin()) return rc;
    const size_t N = c.map.distinct;
    const size_t first = std::min(n_cells, N);
    if (first == 0) return fail(BDG_ERR_ARG, "mean requires at least one data point");
    cudaStream_t st = c.stream;
    const uint32_t* d_distinct = c.map.first_seen();
    const uint32_t* d_counts = c.map.counts();
    if (int e = c.sel_scalars.ensure(64)) return e;
    unsigned long long* d_sum = (unsigned long long*)c.sel_scalars.p;
    uint32_t* d_nsel = (uint32_t*)((char*)c.sel_scalars.p + 8);
    CU_TRY(cudaMemsetAsync(d_sum, 0, 16, st));
    bdg::sum_first_kernel<<<(int)std::min<size_t>((first + 255) / 256, (size_t)c.sms * 4), 256, 0, st>>>(d_counts, (uint32_t)first, d_sum);
    g_launches++;
    unsigned long long sum = 0;
    CU_TRY(cudaMemcpyAsync(&sum, d_sum, 8, cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaStreamSynchronize(st));
    const double cut = std::max(((double)sum / (double)first) / 5.0, 5.0);
    *cutoff = cut;
    const uint32_t thr = (uint32_t)std::floor(cut);          // counts are integers: count > cutoff <=> count > floor(cutoff)
    if (int e = c.sel.ensure(N * 4)) return e;
    thrust::counting_iterator<uint32_t> all(0);
    bdg::CountAbove pred{d_counts, thr};
    size_t tmp = 0;
    CU_TRY(cub::DeviceSelect::If(nullptr, tmp, all, (uint32_t*)c.sel.p, d_nsel, (int)N, pred, st));
    if (int e = c.sel_tmp.ensure(tmp)) return e;
    CU_TRY(cub::DeviceSelect::If(c.sel_tmp.p, tmp, all, (uint32_t*)c.sel.p, d_nsel, (int)N, pred, st));
    uint32_t nsel = 0;
    CU_TRY(cudaMemcpyAsync(&nsel, d_nsel, 4, cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaStreamSynchronize(st));
    *n_above = nsel;
    if (nsel == 0) return BDG_OK;
    if (nsel > cap) return fail(BDG_ERR_CAPACITY, "%u barcodes above the cutoff but room for %zu", nsel, cap);
    if (!top_ranks || !top_counts) return fail(BDG_ERR_ARG, "NULL pointer argument");
    for (Buf* b : {&c.sel_keys, &c.sel_sorted, &c.sel_pos, &c.head_ranks, &c.head_counts}) if (int e = b->ensure((size_t)nsel * 4)) return e;
    if (int e = c.head_hits.ensure(nsel)) return e;
    const uint32_t *sel = (const uint32_t*)c.sel.p, *keys = (const uint32_t*)c.sel_keys.p;
    uint32_t *ranks = (uint32_t*)c.head_ranks.p, *counts = (uint32_t*)c.head_counts.p;
    const int nb = (int)std::min<size_t>(((size_t)nsel + 255) / 256, (size_t)c.sms * 4);
    bdg::centres_keys_kernel<<<nb, 256, 0, st>>>(sel, d_counts, nsel, (uint32_t*)c.sel_keys.p);
    size_t tmp2 = 0;
    CU_TRY(cub::DeviceRadixSort::SortPairs(nullptr, tmp2, keys, (uint32_t*)c.sel_sorted.p, sel, (uint32_t*)c.sel_pos.p, (int)nsel, 0, 32, st));
    if (int e = c.sel_tmp.ensure(tmp2)) return e;
    CU_TRY(cub::DeviceRadixSort::SortPairs(c.sel_tmp.p, tmp2, keys, (uint32_t*)c.sel_sorted.p, sel, (uint32_t*)c.sel_pos.p, (int)nsel, 0, 32, st));
    bdg::centres_gather_kernel<<<nb, 256, 0, st>>>((const uint32_t*)c.sel_pos.p, d_distinct, d_counts, nsel, ranks, counts);
    g_launches += 2;
    CU_TRY(cudaGetLastError());
    if (top_hits) {
        if (W > 0xFFFFFFFFull) return fail(BDG_ERR_ARG, "size exceeds 2^32");
        if (W && !sorted_wl) return fail(BDG_ERR_ARG, "NULL pointer argument");
        const uint32_t* d_wl = sorted_wl;
        if (!wl_on_device) {
            uint32_t* up = nullptr;
            if (int e = stage(c, {piece(up, std::max<size_t>(W, 1) * 4)})) return e;
            CU_TRY(cudaMemcpyAsync(up, sorted_wl, W * 4, cudaMemcpyHostToDevice, st));
            d_wl = up;
        }
        if (int rc = sort_check(c, d_wl, W)) return rc;
        if (int rc = member_sorted_body(d_wl, W, ranks, nsel, (uint8_t*)c.head_hits.p, st)) return rc;
        CU_TRY(cudaMemcpyAsync(top_hits, c.head_hits.p, nsel, cudaMemcpyDeviceToHost, st));
    }
    CU_TRY(cudaMemcpyAsync(top_ranks, ranks, (size_t)nsel * 4, cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaMemcpyAsync(top_counts, counts, (size_t)nsel * 4, cudaMemcpyDeviceToHost, st));
    if (top_hits) return sort_check_result(c);               // (waits for the copies too)
    CU_TRY(cudaStreamSynchronize(st));
    return BDG_OK;
}

static int centres_above_args(unsigned long long token, size_t* n_above, double* cutoff, DevCtx** c)
{
    if (!n_above || !cutoff) return fail(BDG_ERR_ARG, "NULL result pointer");
    *n_above = 0; *cutoff = 0.0;
    return map_ctx(token, c);
}

int bdg_centres_above(unsigned long long token, size_t n_cells, const uint32_t* sorted_wl, size_t W, uint32_t* top_ranks, uint32_t* top_counts,
                      uint8_t* top_hits, size_t cap, size_t* n_above, double* cutoff)
{
    DevCtx* c = nullptr;
    if (int rc = centres_above_args(token, n_above, cutoff, &c)) return rc;
    return centres_above_body(*c, n_cells, sorted_wl, false, W, top_ranks, top_counts, top_hits, cap, n_above, cutoff, c->stream);
}

int bdg_dev_centres_above(unsigned long long token, size_t n_cells, const uint32_t* d_sorted_wl, size_t W, uint32_t* top_ranks,
                          uint32_t* top_counts, uint8_t* top_hits, size_t cap, size_t* n_above, double* cutoff, void* stream)
{
    DevCtx* c = nullptr;
    if (int rc = centres_above_args(token, n_above, cutoff, &c)) return rc;
    if (top_hits && W) if (int rc = check_on_first(d_sorted_wl, "whitelist")) return rc;
    return centres_above_body(*c, n_cells, d_sorted_wl, true, W, top_ranks, top_counts, top_hits, cap, n_above, cutoff, (cudaStream_t)stream);
}

// The stretch of `bc_by_counts` right behind the head bdg_centres_above returns (barcode_graph.py:273-276 runs into it when too few
// centres were found): the first `need` barcodes with count <= floor(cutoff) in count-descending order, ties in first-seen
// order.  One stable stream compaction per count value, from floor(cutoff) downwards, until enough are found.
int bdg_centres_rest(unsigned long long token, double cutoff, size_t need, uint32_t* out_ranks, size_t* n_out)
{
    if (!n_out) return fail(BDG_ERR_ARG, "NULL result pointer");
    *n_out = 0;
    if (need == 0) return BDG_OK;
    if (!out_ranks) return fail(BDG_ERR_ARG, "NULL pointer argument");
    DevCtx* cp = nullptr;
    if (int rc = map_ctx(token, &cp)) return rc;
    DevCtx& c = *cp;
    const size_t N = c.map.distinct;
    cudaStream_t st = c.stream;
    const uint32_t* d_distinct = c.map.first_seen();
    const uint32_t* d_counts = c.map.counts();
    if (int e = c.sel.ensure(N * 4)) return e;
    if (int e = c.head_ranks.ensure(std::min(need, N) * 4)) return e;
    if (int e = c.head_counts.ensure(std::min(need, N) * 4)) return e;
    if (int e = c.sel_scalars.ensure(64)) return e;
    uint32_t* d_nsel = (uint32_t*)((char*)c.sel_scalars.p + 8);
    thrust::counting_iterator<uint32_t> all(0);
    size_t tmp = 0;
    CU_TRY(cub::DeviceSelect::If(nullptr, tmp, all, (uint32_t*)c.sel.p, d_nsel, (int)N, bdg::CountIs{d_counts, 0u}, st));
    if (int e = c.sel_tmp.ensure(tmp)) return e;
    size_t got = 0;
    for (long long v = (long long)std::floor(cutoff); v >= 1 && got < need; v--) {
        CU_TRY(cub::DeviceSelect::If(c.sel_tmp.p, tmp, all, (uint32_t*)c.sel.p, d_nsel, (int)N, bdg::CountIs{d_counts, (uint32_t)v}, st));
        uint32_t nsel = 0;
        CU_TRY(cudaMemcpyAsync(&nsel, d_nsel, 4, cudaMemcpyDeviceToHost, st));
        CU_TRY(cudaStreamSynchronize(st));
        const size_t take = std::min<size_t>(nsel, need - got);
        if (take == 0) continue;
        const int nb = (int)std::min<size_t>((take + 255) / 256, (size_t)c.sms * 4);
        bdg::centres_gather_kernel<<<nb, 256, 0, st>>>((const uint32_t*)c.sel.p, d_distinct, d_counts, (uint32_t)take, (uint32_t*)c.head_ranks.p,
                                                       (uint32_t*)c.head_counts.p);
        g_launches++;
        CU_TRY(cudaMemcpyAsync(out_ranks + got, c.head_ranks.p, take * 4, cudaMemcpyDeviceToHost, st));
        CU_TRY(cudaStreamSynchronize(st));
        got += take;
    }
    *n_out = got;
    return BDG_OK;
}

// ---- f-2  the per-read gather: the 5-byte result per row (centre barcode + "has a centre" byte) ----------------------------
static int assign_reads32_args(unsigned long long token, bool resident, size_t N, const uint32_t* centre_per_row, const uint8_t* has_centre,
                               size_t R_all, size_t* n_assigned, DevCtx** c)
{
    if (n_assigned) *n_assigned = 0;
    if (R_all == 0) return EMPTY;
    if (!centre_per_row || !has_centre) return fail(BDG_ERR_ARG, "NULL pointer argument");
    if (int rc = map_ctx(token, c)) return rc;
    const ReadMap& m = (*c)->map;
    if (N != m.distinct || R_all != m.rows) return fail(BDG_ERR_ARG, "sizes do not match the dedup call the token came from");
    if (resident && N && m.cl_token != m.token) return fail(BDG_ERR_ARG, "no clustering result of this dedup call is resident on the device (bdg_cluster_resident)");
    return BDG_OK;
}

// d_ci (device, on c.dev) is the centre index per node, NULL for the resident clustering result; the 5-byte result goes to d_out /
// d_oh (device, R_all rows), the number of rows with a centre to *n_assigned (optional: the call then waits for it).
static int assign_reads32_body(DevCtx& c, const int32_t* d_ci, size_t N, uint32_t* d_out, uint8_t* d_oh, size_t R_all, size_t* n_assigned,
                               cudaStream_t caller)
{
    CallerOrder order(c, caller);
    if (int rc = order.begin()) return rc;
    cudaStream_t st = c.stream;
    const ReadMap& m = c.map;
    if (int e = c.centre_val.ensure(std::max<size_t>(N, 1) * 5)) return e;
    if (int e = c.counters.ensure(16)) return e;
    if (!d_ci) d_ci = (const int32_t*)m.centre.p;
    CU_TRY(cudaMemsetAsync(c.counters.p, 0, 8, st));
    uint32_t* d_cv = (uint32_t*)c.centre_val.p;
    uint8_t* d_ch = (uint8_t*)c.centre_val.p + std::max<size_t>(N, 1) * 4;
    if (N) {
        const int nb = (int)std::min<size_t>((N + 255) / 256, (size_t)c.sms * 8);
        bdg::centre_of_distinct32_kernel<<<nb, 256, 0, st>>>(d_ci, m.order() /* first-seen -> node */, m.ascending() /* node -> barcode */,
                                                             (uint32_t)N, d_cv, d_ch);
    }
    const int rb = (int)std::min<size_t>((R_all + 255) / 256, (size_t)c.sms * 8);
    bdg::assign_reads32_kernel<<<rb, 256, 0, st>>>(d_cv, d_ch, m.read_pos(), m.masked ? (const uint8_t*)m.valid.p : nullptr,
                                                   m.masked ? (const uint32_t*)m.valid_scan.p : nullptr, (uint32_t)R_all, d_out, d_oh,
                                                   (unsigned long long*)c.counters.p);
    g_launches += 2;
    CU_TRY(cudaGetLastError());
    if (n_assigned) {
        unsigned long long cnt = 0;
        CU_TRY(cudaMemcpyAsync(&cnt, c.counters.p, 8, cudaMemcpyDeviceToHost, st));
        CU_TRY(cudaStreamSynchronize(st));
        *n_assigned = (size_t)cnt;
    }
    return BDG_OK;
}

// centre_idx == NULL: the clustering a bdg_cluster_resident call left on the device is used in place (nothing is uploaded).
int bdg_assign_reads32(unsigned long long token, const int32_t* centre_idx, size_t N, uint32_t* centre_per_row, uint8_t* has_centre, size_t R_all,
                       size_t* n_assigned)
{
    DevCtx* c = nullptr;
    if (int rc = assign_reads32_args(token, !centre_idx, N, centre_per_row, has_centre, R_all, n_assigned, &c)) return done(rc);
    cudaStream_t st = c->stream;
    int32_t* d_ci = nullptr;
    uint32_t* d_out = nullptr;
    uint8_t* d_oh = nullptr;
    if (int e = stage(*c, {piece(d_out, R_all * 4), piece(d_oh, R_all), piece(d_ci, centre_idx ? N * 4 : 0)})) return e;
    if (centre_idx) CU_TRY(cudaMemcpyAsync(d_ci, centre_idx, N * 4, cudaMemcpyHostToDevice, st));
    if (int rc = assign_reads32_body(*c, centre_idx ? d_ci : nullptr, N, d_out, d_oh, R_all, n_assigned, st)) return rc;
    CU_TRY(cudaMemcpyAsync(centre_per_row, d_out, R_all * 4, cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaMemcpyAsync(has_centre, d_oh, R_all, cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaStreamSynchronize(st));
    return BDG_OK;
}

int bdg_dev_assign_reads32(unsigned long long token, const int32_t* d_centre_idx, size_t N, uint32_t* d_centre_per_row, uint8_t* d_has_centre,
                           size_t R_all, size_t* n_assigned, void* stream)
{
    DevCtx* c = nullptr;
    if (int rc = assign_reads32_args(token, !d_centre_idx, N, d_centre_per_row, d_has_centre, R_all, n_assigned, &c)) return done(rc);
    if (d_centre_idx && N) if (int rc = check_on_first(d_centre_idx, "centre_idx")) return rc;
    if (int rc = check_on_first(d_centre_per_row, "centre_per_row")) return rc;
    if (int rc = check_on_first(d_has_centre, "has_centre")) return rc;
    return assign_reads32_body(*c, N ? d_centre_idx : nullptr, N, d_centre_per_row, d_has_centre, R_all, n_assigned, (cudaStream_t)stream);
}

// The per-read gather for rows outside any read map: every valid row's barcode is looked up among the token's nodes (the
// ascending array).
static int assign_lookup32_args(unsigned long long token, bool resident, size_t N, const uint32_t* ranks, size_t R, const uint32_t* centre,
                                const uint8_t* has_centre, size_t* n_assigned, size_t* n_missing, DevCtx** c)
{
    if (n_assigned) *n_assigned = 0;
    if (n_missing) *n_missing = 0;
    if (int rc = map_ctx(token, c)) return rc;
    const ReadMap& m = (*c)->map;
    if (N != m.distinct) return fail(BDG_ERR_ARG, "N does not match the read map the token names");
    if (resident && m.cl_token != m.token) return fail(BDG_ERR_ARG, "no clustering result of this read map is resident on the device (bdg_cluster_resident)");
    if (R == 0) return EMPTY;
    if (!ranks || !centre || !has_centre) return fail(BDG_ERR_ARG, "NULL pointer argument");
    return BDG_OK;
}

// d_ci as for assign_reads32_body; the counters (assigned, missing) go to *n_assigned / *n_missing (optional: the call then waits).
static int assign_lookup32_body(DevCtx& c, const int32_t* d_ci, size_t N, const uint32_t* d_ranks, const uint8_t* d_valid, size_t R,
                                uint32_t* d_out, uint8_t* d_oh, size_t* n_assigned, size_t* n_missing, cudaStream_t caller)
{
    CallerOrder order(c, caller);
    if (int rc = order.begin()) return rc;
    cudaStream_t st = c.stream;
    if (int e = c.counters.ensure(16)) return e;
    if (!d_ci) d_ci = (const int32_t*)c.map.centre.p;
    CU_TRY(cudaMemsetAsync(c.counters.p, 0, 16, st));
    const int rb = (int)std::min<size_t>((R + bdg::NT - 1) / bdg::NT, (size_t)c.sms * 8);
    bdg::lookup_assign32_kernel<<<rb, bdg::NT, 0, st>>>(c.map.ascending(), (uint32_t)N, d_ci, d_ranks, d_valid, R, d_out, d_oh,
                                                         (unsigned long long*)c.counters.p);
    g_launches++;
    CU_TRY(cudaGetLastError());
    if (n_assigned || n_missing) {
        unsigned long long cnt[2] = {0, 0};
        CU_TRY(cudaMemcpyAsync(cnt, c.counters.p, 16, cudaMemcpyDeviceToHost, st));
        CU_TRY(cudaStreamSynchronize(st));
        if (n_assigned) *n_assigned = (size_t)cnt[0];
        if (n_missing) *n_missing = (size_t)cnt[1];
    }
    return BDG_OK;
}

int bdg_assign_lookup32(unsigned long long token, const int32_t* centre_idx, size_t N, const uint32_t* ranks, const uint8_t* valid, size_t R,
                        uint32_t* centre, uint8_t* has_centre, size_t* n_assigned, size_t* n_missing)
{
    DevCtx* c = nullptr;
    if (int rc = assign_lookup32_args(token, !centre_idx, N, ranks, R, centre, has_centre, n_assigned, n_missing, &c)) return done(rc);
    cudaStream_t st = c->stream;
    uint32_t *d_ranks = nullptr, *d_out = nullptr;
    uint8_t *d_valid = nullptr, *d_oh = nullptr;
    int32_t* d_ci = nullptr;
    if (int e = stage(*c, {piece(d_ranks, R * 4), piece(d_valid, valid ? R : 0), piece(d_out, R * 4), piece(d_oh, R),
                           piece(d_ci, centre_idx ? N * 4 : 0)})) return e;
    CU_TRY(cudaMemcpyAsync(d_ranks, ranks, R * 4, cudaMemcpyHostToDevice, st));
    if (valid) CU_TRY(cudaMemcpyAsync(d_valid, valid, R, cudaMemcpyHostToDevice, st));
    if (centre_idx) CU_TRY(cudaMemcpyAsync(d_ci, centre_idx, N * 4, cudaMemcpyHostToDevice, st));
    if (int rc = assign_lookup32_body(*c, centre_idx ? d_ci : nullptr, N, d_ranks, valid ? d_valid : nullptr, R, d_out, d_oh, n_assigned,
                                      n_missing, st)) return rc;
    CU_TRY(cudaMemcpyAsync(centre, d_out, R * 4, cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaMemcpyAsync(has_centre, d_oh, R, cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaStreamSynchronize(st));
    return BDG_OK;
}

int bdg_dev_assign_lookup32(unsigned long long token, const int32_t* d_centre_idx, size_t N, const uint32_t* d_ranks, const uint8_t* d_valid,
                            size_t R, uint32_t* d_centre, uint8_t* d_has_centre, size_t* n_assigned, size_t* n_missing, void* stream)
{
    DevCtx* c = nullptr;
    if (int rc = assign_lookup32_args(token, !d_centre_idx, N, d_ranks, R, d_centre, d_has_centre, n_assigned, n_missing, &c)) return done(rc);
    if (d_centre_idx) if (int rc = check_on_first(d_centre_idx, "centre_idx")) return rc;
    if (int rc = check_on_first(d_ranks, "ranks")) return rc;
    if (d_valid) if (int rc = check_on_first(d_valid, "valid")) return rc;
    if (int rc = check_on_first(d_centre, "centre")) return rc;
    if (int rc = check_on_first(d_has_centre, "has_centre")) return rc;
    return assign_lookup32_body(*c, d_centre_idx, N, d_ranks, d_valid, R, d_centre, d_has_centre, n_assigned, n_missing, (cudaStream_t)stream);
}

int bdg_pack16(const char* seqs, size_t R, uint32_t* out, uint8_t* valid)
{
    if (R == 0) return BDG_OK;
    if (!seqs || !out || !valid) return fail(BDG_ERR_ARG, "NULL pointer argument");
    DevCtx* c = nullptr;
    if (int rc = first_ctx(&c)) return rc;
    char* d_seqs = nullptr;
    uint32_t* d_out = nullptr;
    uint8_t* d_valid = nullptr;
    if (int e = stage(*c, {piece(d_seqs, R * 16), piece(d_out, R * 4), piece(d_valid, R)})) return e;
    CU_TRY(cudaMemcpyAsync(d_seqs, seqs, R * 16, cudaMemcpyHostToDevice, c->stream));
    if (int rc = bdg_dev_pack16(d_seqs, R, d_out, d_valid, c->stream)) return rc;
    CU_TRY(cudaMemcpyAsync(out, d_out, R * 4, cudaMemcpyDeviceToHost, c->stream));
    CU_TRY(cudaMemcpyAsync(valid, d_valid, R, cudaMemcpyDeviceToHost, c->stream));
    CU_TRY(cudaStreamSynchronize(c->stream));
    return BDG_OK;
}

// badger.py:82-88 for the array pipeline: the whitelist records packed (a-1), the invalid ones dropped, sorted and made
// distinct on the device (cub radix sort + unique); out_sorted has room for R entries, *n receives the number kept.
static int pack16_sorted_args(const char* seqs, size_t R, const uint32_t* out_sorted, size_t* n, DevCtx** c)
{
    if (!n) return fail(BDG_ERR_ARG, "NULL result pointer");
    *n = 0;
    if (R == 0) return EMPTY;
    if (!seqs || !out_sorted) return fail(BDG_ERR_ARG, "NULL pointer argument");
    if (R > 0x7FFFFFFFull) return fail(BDG_ERR_ARG, "more than 2^31 records in one call");
    return first_ctx(c);
}

// d_seqs: the R records on c.dev; ranks / valid: scratch for R entries; the distinct packed barcodes are copied to out_sorted
// (kind: to the host or to device memory on c.dev; the host form waits for the copy).
static int pack16_sorted_body(DevCtx& c, const char* d_seqs, size_t R, uint32_t* ranks, uint8_t* valid, uint32_t* out_sorted, cudaMemcpyKind kind,
                              size_t* n, cudaStream_t caller)
{
    CallerOrder order(c, caller);
    if (int rc = order.begin()) return rc;
    cudaStream_t st = c.stream;
    for (Buf* b : {&c.sel, &c.sel_keys, &c.sel_sorted}) if (int e = b->ensure(R * 4)) return e;
    if (int e = c.sel_scalars.ensure(64)) return e;
    uint32_t *kept_ranks = (uint32_t*)c.sel.p, *sorted = (uint32_t*)c.sel_keys.p, *distinct = (uint32_t*)c.sel_sorted.p;
    uint32_t* d_n = (uint32_t*)c.sel_scalars.p;
    if (int rc = bdg_dev_pack16(d_seqs, R, ranks, valid, st)) return rc;
    size_t t1 = 0, t2 = 0, t3 = 0;
    CU_TRY(cub::DeviceSelect::Flagged(nullptr, t1, (const uint32_t*)ranks, (const uint8_t*)valid, kept_ranks, d_n, (int)R, st));
    CU_TRY(cub::DeviceRadixSort::SortKeys(nullptr, t2, (const uint32_t*)kept_ranks, sorted, (int)R, 0, 32, st));
    CU_TRY(cub::DeviceSelect::Unique(nullptr, t3, (const uint32_t*)sorted, distinct, d_n, (int)R, st));
    if (int e = c.sel_tmp.ensure(std::max(t1, std::max(t2, t3)))) return e;
    CU_TRY(cub::DeviceSelect::Flagged(c.sel_tmp.p, t1, (const uint32_t*)ranks, (const uint8_t*)valid, kept_ranks, d_n, (int)R, st));
    uint32_t kept = 0;
    CU_TRY(cudaMemcpyAsync(&kept, d_n, 4, cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaStreamSynchronize(st));
    if (kept == 0) return BDG_OK;
    CU_TRY(cub::DeviceRadixSort::SortKeys(c.sel_tmp.p, t2, (const uint32_t*)kept_ranks, sorted, (int)kept, 0, 32, st));
    CU_TRY(cub::DeviceSelect::Unique(c.sel_tmp.p, t3, (const uint32_t*)sorted, distinct, d_n, (int)kept, st));
    uint32_t n_distinct = 0;
    CU_TRY(cudaMemcpyAsync(&n_distinct, d_n, 4, cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaStreamSynchronize(st));
    CU_TRY(cudaMemcpyAsync(out_sorted, distinct, (size_t)n_distinct * 4, kind, st));
    if (kind == cudaMemcpyDeviceToHost) CU_TRY(cudaStreamSynchronize(st));
    *n = n_distinct;
    return BDG_OK;
}

int bdg_pack16_sorted(const char* seqs, size_t R, uint32_t* out_sorted, size_t* n)
{
    DevCtx* c = nullptr;
    if (int rc = pack16_sorted_args(seqs, R, out_sorted, n, &c)) return done(rc);
    char* d_seqs = nullptr;
    uint32_t* ranks = nullptr;
    uint8_t* valid = nullptr;
    if (int e = stage(*c, {piece(d_seqs, R * 16), piece(ranks, R * 4), piece(valid, R)})) return e;
    CU_TRY(cudaMemcpyAsync(d_seqs, seqs, R * 16, cudaMemcpyHostToDevice, c->stream));
    return pack16_sorted_body(*c, d_seqs, R, ranks, valid, out_sorted, cudaMemcpyDeviceToHost, n, c->stream);
}

int bdg_dev_pack16_sorted(const char* d_seqs, size_t R, uint32_t* d_out_sorted, size_t* n, void* stream)
{
    DevCtx* c = nullptr;
    if (int rc = pack16_sorted_args(d_seqs, R, d_out_sorted, n, &c)) return done(rc);
    if (int rc = check_on_first(d_seqs, "records")) return rc;
    if (int rc = check_on_first(d_out_sorted, "out_sorted")) return rc;
    uint32_t* ranks = nullptr;
    uint8_t* valid = nullptr;
    if (int e = stage(*c, {piece(ranks, R * 4), piece(valid, R)})) return e;
    return pack16_sorted_body(*c, d_seqs, R, ranks, valid, d_out_sorted, cudaMemcpyDeviceToDevice, n, (cudaStream_t)stream);
}

// One device's share of a host-buffer edge build: upload, launch, read the count back (re-run once with the exact
// size when the guess was too small).  Runs on its own host thread when several devices take part, because the
// sparse passes read a tile count back between their kernels.
// src_dev < 0: `sorted` is a host array; else it lives on device src_dev (peer copy over NVLink, or nothing to copy at all
// when that is this device's own workspace).
static int edges_on_device(DevCtx& c, const uint32_t* sorted, size_t N, int t, int part, int nparts, size_t* n_out, int src_dev = -1)
{
    CU_TRY(cudaSetDevice(c.dev));
    if (int e = c.sorted.ensure(std::max<size_t>(N, 1) * 4)) return e;
    if (int e = c.count.ensure(2 * sizeof(unsigned long long))) return e;      // [edge count | first unsorted index]
    if (src_dev < 0) CU_TRY(cudaMemcpyAsync(c.sorted.p, sorted, N * 4, cudaMemcpyHostToDevice, c.stream));
    else if (src_dev == c.dev) CU_TRY(cudaMemcpyAsync(c.sorted.p, sorted, N * 4, cudaMemcpyDeviceToDevice, c.stream));
    else CU_TRY(cudaMemcpyPeerAsync(c.sorted.p, c.dev, sorted, src_dev, N * 4, c.stream));
    // the input must be strictly increasing: checked on the device, read back together with the edge count
    unsigned long long* d_bad = (unsigned long long*)c.count.p + 1;
    unsigned long long first_bad = ~0ull;
    CU_TRY(cudaMemsetAsync(d_bad, 0xFF, 8, c.stream));
    if (N > 1) {
        bdg::sorted_check_kernel<true><<<(int)std::min<size_t>((N + 255) / 256, (size_t)c.sms * 8), 256, 0, c.stream>>>((const uint32_t*)c.sorted.p, (uint32_t)N, d_bad);
        g_launches++;
    }
    size_t cap = std::max(edge_cap_guess(N, t, nparts), c.ea.cap / 4);
    unsigned long long count = 0;
    bool done = false;
    for (int attempt = 0; attempt < 4 && !done; attempt++) {
        if (int e = c.ea.ensure(cap * 4)) return e;
        if (int e = c.eb.ensure(cap * 4)) return e;
        if (int e = c.ed.ensure(cap)) return e;
        if (int e = launch_edges((const uint32_t*)c.sorted.p, N, t, part, nparts, (uint32_t*)c.ea.p, (uint32_t*)c.eb.p, (uint8_t*)c.ed.p, cap,
                                 (unsigned long long*)c.count.p, c.stream, &c)) return e;
        unsigned long long both[2] = {0, 0};
        CU_TRY(cudaMemcpyAsync(both, c.count.p, sizeof(both), cudaMemcpyDeviceToHost, c.stream));
        CU_TRY(cudaStreamSynchronize(c.stream));
        count = both[0];
        first_bad = both[1];
        if (first_bad != ~0ull) return fail(BDG_ERR_ARG, "input not strictly increasing at index %llu", first_bad);
        if (count >> 63) {                     // rare: a sparse pass listed more tiles than the list holds; grow it and run again
            if (int e = grow_tile_lists(c)) return e;
        } else if (count > cap) {              // rare: the capacity guess was too small; the edge set is deterministic, so run again
            cap = (size_t)count;
        } else {
            done = true;
        }
    }
    if (!done) return fail(BDG_ERR_CUDA, "edge construction did not settle after growing its buffers (count %llu)", count);
    c.generation++;
    *n_out = (size_t)count;
    return BDG_OK;
}

static int edges_on_devices(const uint32_t* sorted, size_t N, int t, const std::vector<int>& ctx_idx,
                            const std::vector<int>& parts, int nparts, bdg_edges* res, int src_dev = -1)
{
    const double t0 = now_ms();
    const size_t G = ctx_idx.size();
    std::vector<int> rcs(G, BDG_OK);
    std::vector<std::string> errs(G);
    std::vector<size_t> counts(G, 0);
    std::vector<double> took(G, 0.0);
    auto work = [&](size_t g) {
        const double w0 = now_ms();
        rcs[g] = edges_on_device(g_ctx[ctx_idx[g]], sorted, N, t, parts[g], nparts, &counts[g], src_dev);
        took[g] = now_ms() - w0;
        if (rcs[g]) errs[g] = g_err;       // g_err is thread-local
    };
    if (G == 1) work(0);
    else {
        std::vector<std::thread> th;
        for (size_t g = 0; g < G; g++) th.emplace_back(work, g);
        for (auto& x : th) x.join();
    }
    if (!g_ctx.empty()) cudaSetDevice(g_ctx[0].dev);
    for (size_t g = 0; g < G; g++)
        if (rcs[g]) return fail(rcs[g], "%s", errs[g].c_str());
    size_t total = 0;
    for (size_t g = 0; g < G; g++) {
        res->ctx.push_back(ctx_idx[g]);
        res->count.push_back(counts[g]);
        res->gen.push_back(g_ctx[ctx_idx[g]].generation);
        total += counts[g];
    }
    if (getenv("BDG_TRACE")) {
        fprintf(stderr, "[bdg] edges N=%zu t=%d devices=%zu: upload + kernels %.2f ms, edges %zu; per device (ms / edges):", N, t, G, now_ms() - t0, total);
        for (size_t g = 0; g < G; g++) fprintf(stderr, " %.1f/%zu", took[g], counts[g]);
        fprintf(stderr, "\n");
    }
    return BDG_OK;
}

int bdg_edges_build(const uint32_t* sorted_unique, size_t N, int t, bdg_edges** out)
{
    if (!out || (N && !sorted_unique)) return fail(BDG_ERR_ARG, "NULL pointer argument");
    *out = nullptr;
    if (int rc = need_ctx()) return rc;                    // (the strictly-increasing check runs on the device)
    bdg_edges* res = new (std::nothrow) bdg_edges();
    if (!res) return fail(BDG_ERR_OOM, "host allocation failed");
    std::vector<int> idx, parts;
    const int G = (int)g_ctx.size();
    for (int g = 0; g < G; g++) { idx.push_back(g); parts.push_back(g); }
    int rc = BDG_OK;
    try { rc = edges_on_devices(sorted_unique, N, t, idx, parts, G, res); }
    catch (const std::bad_alloc&) { rc = fail(BDG_ERR_OOM, "host allocation failed"); }
    catch (const std::exception& e) { rc = fail(BDG_ERR_CUDA, "host thread failure: %s", e.what()); }
    if (rc) { delete res; return rc; }
    *out = res;
    return BDG_OK;
}

// The same over the ascending distinct barcodes a bdg_dedup_reads call left on the first device: nothing is uploaded, the other
// devices fetch the array with peer copies.
int bdg_edges_build_resident(unsigned long long token, int t, bdg_edges** out)
{
    if (!out) return fail(BDG_ERR_ARG, "NULL pointer argument");
    *out = nullptr;
    DevCtx* c0 = nullptr;
    if (int rc = map_ctx(token, &c0)) return rc;
    bdg_edges* res = new (std::nothrow) bdg_edges();
    if (!res) return fail(BDG_ERR_OOM, "host allocation failed");
    res->read_map = token;
    std::vector<int> idx, parts;
    const int G = (int)g_ctx.size();
    for (int g = 0; g < G; g++) { idx.push_back(g); parts.push_back(g); }
    int rc = BDG_OK;
    try { rc = edges_on_devices(c0->map.ascending(), c0->map.distinct, t, idx, parts, G, res, c0->dev); }
    catch (const std::bad_alloc&) { rc = fail(BDG_ERR_OOM, "host allocation failed"); }
    catch (const std::exception& e) { rc = fail(BDG_ERR_CUDA, "host thread failure: %s", e.what()); }
    if (rc) { delete res; return rc; }
    *out = res;
    return BDG_OK;
}

// One part's edges straight into caller buffers of `cap` entries each (page-locked ones copy at PCIe speed): with the join
// form the finished edges of earlier seed conditions cross PCIe while later ones are still being joined.  *count receives the
// number of edges found; when it exceeds cap only the first cap were stored and the call has to be repeated with more room.
int bdg_edges_build_into(const uint32_t* sorted_unique, size_t N, int t, int part, int nparts, uint32_t* a, uint32_t* b, uint8_t* d, size_t cap,
                         size_t* count)
{
    if (!count || (N && !sorted_unique) || (cap && (!a || !b || !d))) return fail(BDG_ERR_ARG, "NULL pointer argument");
    *count = 0;
    if (nparts < 1 || part < 0 || part >= nparts) return fail(BDG_ERR_ARG, "part %d of %d is not a valid part", part, nparts);
    if (int rc = need_ctx()) return rc;
    DevCtx& c = g_ctx[0];
    CU_TRY(cudaSetDevice(c.dev));
    const size_t dcap = std::max<size_t>(cap, 1);
    if (int e = c.sorted.ensure(std::max<size_t>(N, 1) * 4)) return e;
    if (int e = c.count.ensure(2 * sizeof(unsigned long long))) return e;
    if (int e = c.ea.ensure(dcap * 4)) return e;
    if (int e = c.eb.ensure(dcap * 4)) return e;
    if (int e = c.ed.ensure(dcap)) return e;
    c.generation++;                                         // older handles on this device lose their edges
    CU_TRY(cudaMemcpyAsync(c.sorted.p, sorted_unique, N * 4, cudaMemcpyHostToDevice, c.stream));
    unsigned long long* d_bad = (unsigned long long*)c.count.p + 1;
    CU_TRY(cudaMemsetAsync(d_bad, 0xFF, 8, c.stream));
    if (N > 1) {
        bdg::sorted_check_kernel<true><<<(int)std::min<size_t>((N + 255) / 256, (size_t)c.sms * 8), 256, 0, c.stream>>>((const uint32_t*)c.sorted.p, (uint32_t)N, d_bad);
        g_launches++;
    }
    const bool streaming = t > 0 && N >= 2 && edge_mode_for(t, N) == 2;
    JoinStream js{a, b, d, cap};
    for (int attempt = 0; attempt < 3; attempt++) {
        if (int e = launch_edges((const uint32_t*)c.sorted.p, N, t, part, nparts, (uint32_t*)c.ea.p, (uint32_t*)c.eb.p, (uint8_t*)c.ed.p, cap,
                                 (unsigned long long*)c.count.p, c.stream, &c, streaming ? &js : nullptr)) return e;
        unsigned long long both[2] = {0, 0};
        CU_TRY(cudaMemcpyAsync(both, c.count.p, sizeof(both), cudaMemcpyDeviceToHost, c.stream));
        CU_TRY(cudaStreamSynchronize(c.stream));
        if (both[1] != ~0ull) return fail(BDG_ERR_ARG, "input not strictly increasing at index %llu", both[1]);
        if (both[0] >> 63) {                                // a sparse pass listed more tiles than its list holds: grow it and run again
            if (int e = grow_tile_lists(c)) return e;
            continue;
        }
        *count = (size_t)both[0];
        if (!streaming) {
            const size_t k = std::min<size_t>(*count, cap);
            if (k) {
                CU_TRY(cudaMemcpyAsync(a, c.ea.p, k * 4, cudaMemcpyDeviceToHost, c.stream));
                CU_TRY(cudaMemcpyAsync(b, c.eb.p, k * 4, cudaMemcpyDeviceToHost, c.stream));
                CU_TRY(cudaMemcpyAsync(d, c.ed.p, k, cudaMemcpyDeviceToHost, c.stream));
                CU_TRY(cudaStreamSynchronize(c.stream));
            }
        }
        return BDG_OK;
    }
    return fail(BDG_ERR_CUDA, "edge construction did not settle after growing its tile lists");
}

int bdg_edges_build_part(const uint32_t* sorted_unique, size_t N, int t, int part, int nparts, bdg_edges** out)
{
    if (!out || (N && !sorted_unique)) return fail(BDG_ERR_ARG, "NULL pointer argument");
    *out = nullptr;
    if (nparts < 1 || part < 0 || part >= nparts) return fail(BDG_ERR_ARG, "part %d of %d is not a valid part", part, nparts);
    if (int rc = need_ctx()) return rc;
    bdg_edges* res = new (std::nothrow) bdg_edges();
    if (!res) return fail(BDG_ERR_OOM, "host allocation failed");
    int rc = BDG_OK;
    try { rc = edges_on_devices(sorted_unique, N, t, {0}, {part}, nparts, res); }
    catch (const std::bad_alloc&) { rc = fail(BDG_ERR_OOM, "host allocation failed"); }
    if (rc) { delete res; return rc; }
    *out = res;
    return BDG_OK;
}

size_t bdg_edges_count(const bdg_edges* e)
{
    size_t n = 0;
    if (e) for (size_t c : e->count) n += c;
    return n;
}

static int check_edges_handle(const bdg_edges* e)
{
    for (size_t g = 0; g < e->ctx.size(); g++)
        if (e->ctx[g] < 0 || (size_t)e->ctx[g] >= g_ctx.size() || g_ctx[e->ctx[g]].generation != e->gen[g])
            return fail(BDG_ERR_ARG, "stale edge handle: a later edge build on the same device has reused its buffers");
    return BDG_OK;
}

int bdg_edges_copy(const bdg_edges* e, uint32_t* a, uint32_t* b, uint8_t* d)
{
    if (!e) return fail(BDG_ERR_ARG, "NULL edge handle");
    const size_t n = bdg_edges_count(e);
    if (n && (!a || !b || !d)) return fail(BDG_ERR_ARG, "NULL output pointer");
    if (int rc = check_edges_handle(e)) return rc;
    const double tc0 = now_ms();
    size_t off = 0;
    for (size_t g = 0; g < e->ctx.size(); g++) {
        DevCtx& c = g_ctx[e->ctx[g]];
        const size_t k = e->count[g];
        if (k) {
            CU_TRY(cudaSetDevice(c.dev));
            CU_TRY(cudaMemcpyAsync(a + off, c.ea.p, k * 4, cudaMemcpyDeviceToHost, c.stream));
            CU_TRY(cudaMemcpyAsync(b + off, c.eb.p, k * 4, cudaMemcpyDeviceToHost, c.stream));
            CU_TRY(cudaMemcpyAsync(d + off, c.ed.p, k, cudaMemcpyDeviceToHost, c.stream));
        }
        off += k;
    }
    for (size_t g = 0; g < e->ctx.size(); g++)
        if (e->count[g]) { CU_TRY(cudaSetDevice(g_ctx[e->ctx[g]].dev)); CU_TRY(cudaStreamSynchronize(g_ctx[e->ctx[g]].stream)); }
    if (!g_ctx.empty()) cudaSetDevice(g_ctx[0].dev);
    if (getenv("BDG_TRACE")) fprintf(stderr, "[bdg] edges_copy %zu edges %.3f ms\n", n, now_ms() - tc0);
    return BDG_OK;
}

// Every part is copied on the first device's stream (peer copies for parts on other devices; the builds have finished when the
// handle is returned).  The part's own stream then waits for the copy too, so that a later build there cannot overwrite the
// edges while they are still being read.
int bdg_dev_edges_copy(const bdg_edges* e, uint32_t* d_a, uint32_t* d_b, uint8_t* d_d, void* stream)
{
    if (!e) return fail(BDG_ERR_ARG, "NULL edge handle");
    const size_t n = bdg_edges_count(e);
    if (n && (!d_a || !d_b || !d_d)) return fail(BDG_ERR_ARG, "NULL output pointer");
    if (int rc = check_edges_handle(e)) return rc;
    if (n == 0) return BDG_OK;
    DevCtx& c0 = g_ctx[0];
    CU_TRY(cudaSetDevice(c0.dev));
    if (int rc = check_on_first(d_a, "a")) return rc;
    if (int rc = check_on_first(d_b, "b")) return rc;
    if (int rc = check_on_first(d_d, "d")) return rc;
    CallerOrder order(c0, stream);
    if (int rc = order.begin()) return rc;
    size_t off = 0;
    for (size_t g = 0; g < e->ctx.size(); g++) {
        DevCtx& c = g_ctx[e->ctx[g]];
        const size_t k = e->count[g];
        if (k) {
            CU_TRY(cudaMemcpyPeerAsync(d_a + off, c0.dev, c.ea.p, c.dev, k * 4, c0.stream));
            CU_TRY(cudaMemcpyPeerAsync(d_b + off, c0.dev, c.eb.p, c.dev, k * 4, c0.stream));
            CU_TRY(cudaMemcpyPeerAsync(d_d + off, c0.dev, c.ed.p, c.dev, k, c0.stream));
        }
        off += k;
    }
    CU_TRY(cudaEventRecord(c0.ev_caller, c0.stream));
    for (size_t g = 0; g < e->ctx.size(); g++) {
        DevCtx& c = g_ctx[e->ctx[g]];
        if (e->count[g] && &c != &c0) CU_TRY(cudaStreamWaitEvent(c.stream, c0.ev_caller, 0));
    }
    return BDG_OK;
}

void bdg_edges_free(bdg_edges* e) { delete e; }


// ---- f-3  cluster(): barcode_graph.py:279-301 -------------------------------------------------------------
// d_ea / d_eb hold barcode VALUES on entry and node indices on return (converted in place).
// centre_idx / level may be NULL: the result then only stays on the device (map.centre / map.level) for bdg_assign_reads*.
// The phases of cluster() over node arrays the caller owns, each on the stream it is given: cluster_on_device runs them on one
// device; the bdg_dev_cluster_* entry points expose them to one process per GPU, which reduces the claims between the ranks.
// values -> node indices of the E edges (ea, eb) against d_sorted[N] on device c (top16: its search table), written to (oa, ob)
static int index_edges(DevCtx& c, const uint32_t* d_sorted, size_t N, const uint32_t* d_ea, const uint32_t* d_eb, size_t E, uint32_t* d_oa,
                       uint32_t* d_ob, cudaStream_t st)
{
    if (int e = c.top16.ensure(65537 * 4)) return e;
    const int nb = (int)std::min<size_t>((N + 256) / 256, (size_t)c.sms * 8);
    bdg::top_start_kernel<<<nb, 256, 0, st>>>(d_sorted, (uint32_t)N, (uint32_t*)c.top16.p);
    if (E) {
        const int eb = (int)std::min<size_t>((E + 255) / 256, (size_t)c.sms * 16);
        bdg::cluster_index_kernel<<<eb, 256, 0, st>>>(d_sorted, (const uint32_t*)c.top16.p, d_ea, d_eb, E, d_oa, d_ob);
    }
    g_launches += 2;
    CU_TRY(cudaGetLastError());
    return BDG_OK;
}

static int node_blocks(size_t N, int sms) { return (int)std::min<size_t>((N + 255) / 256, (size_t)sms * 8); }
static int edge_blocks(size_t E, int sms) { return (int)std::min<size_t>((E + 255) / 256, (size_t)sms * 16); }

// every node free (centre -2, level 255, no claim), then the centres (barcode values d_cen[C]; unobserved ones have no node) seeded
static int cluster_init(const uint32_t* d_sorted, size_t N, const uint32_t* d_cen, size_t C, int32_t* d_ci, uint8_t* d_lv, int32_t* d_min,
                        int32_t* d_max, int sms, cudaStream_t st)
{
    bdg::cluster_init_kernel<<<node_blocks(N, sms), 256, 0, st>>>(d_ci, d_lv, d_min, d_max, (uint32_t)N);
    if (C) bdg::cluster_seed_kernel<<<node_blocks(C, sms), 256, 0, st>>>(d_sorted, (uint32_t)N, d_cen, (uint32_t)C, d_ci, d_lv);
    g_launches += 2;
    CU_TRY(cudaGetLastError());
    return BDG_OK;
}

static int cluster_mark(const uint32_t* d_ia, const uint32_t* d_ib, size_t E, uint8_t* d_lv, unsigned int* d_bad, int sms, cudaStream_t st)
{
    if (E == 0) return BDG_OK;
    bdg::cluster_mark_kernel<<<edge_blocks(E, sms), 256, 0, st>>>(d_ia, d_ib, E, d_lv, d_bad);
    g_launches++;
    CU_TRY(cudaGetLastError());
    return BDG_OK;
}

static int cluster_claim(const uint32_t* d_ia, const uint32_t* d_ib, size_t E, int round, const int32_t* d_ci, const uint8_t* d_lv, int32_t* d_min,
                         int32_t* d_max, int sms, cudaStream_t st)
{
    if (E == 0) return BDG_OK;
    bdg::cluster_claim_kernel<<<edge_blocks(E, sms), 256, 0, st>>>(d_ia, d_ib, E, round, d_ci, d_lv, d_min, d_max);
    g_launches++;
    CU_TRY(cudaGetLastError());
    return BDG_OK;
}

static int cluster_resolve(int32_t* d_ci, uint8_t* d_lv, int32_t* d_min, int32_t* d_max, size_t N, int round, int sms, cudaStream_t st)
{
    bdg::cluster_resolve_kernel<<<node_blocks(N, sms), 256, 0, st>>>(d_ci, d_lv, d_min, d_max, (uint32_t)N, round);
    g_launches++;
    CU_TRY(cudaGetLastError());
    return BDG_OK;
}

// d_ea / d_eb hold barcode VALUES on entry and node indices on return (converted in place) unless `indexed`.
// centre_idx / level may be NULL: the result then only stays on the device (map.centre / map.level) for bdg_assign_reads*.
static int cluster_on_device(DevCtx& c, const uint32_t* d_sorted, size_t N, uint32_t* d_ea, uint32_t* d_eb, size_t E,
                             const uint32_t* centres, size_t C, int rounds, int32_t* centre_idx, uint8_t* level, size_t* n_has_edge = nullptr,
                             bool indexed = false)
{
    cudaStream_t st = c.stream;
    c.map.cl_token = 0;                                    // the resident result is about to be overwritten
    if (int e = c.cl_centres.ensure(std::max<size_t>(C, 1) * 4)) return e;
    if (int e = c.map.centre.ensure(N * 4)) return e;
    if (int e = c.map.level.ensure(N)) return e;
    if (int e = c.cl_min.ensure(N * 4)) return e;
    if (int e = c.cl_max.ensure(N * 4)) return e;
    if (int e = c.cl_flags.ensure(16)) return e;
    unsigned int* d_bad = (unsigned int*)c.cl_flags.p;
    CU_TRY(cudaMemsetAsync(d_bad, 0, 4, c.stream));
    uint32_t* d_cen = (uint32_t*)c.cl_centres.p;
    int32_t *d_ci = (int32_t*)c.map.centre.p, *d_min = (int32_t*)c.cl_min.p, *d_max = (int32_t*)c.cl_max.p;
    uint8_t* d_lv = (uint8_t*)c.map.level.p;
    const int nb = node_blocks(N, c.sms);
    const bool trace = getenv("BDG_TRACE") != nullptr;
    double tr0 = 0, tr1 = 0, tr2 = 0;
    if (trace) { cudaStreamSynchronize(st); tr0 = now_ms(); }
    CU_TRY(cudaMemcpyAsync(d_cen, centres, C * 4, cudaMemcpyHostToDevice, st));
    if (int rc = cluster_init(d_sorted, N, d_cen, C, d_ci, d_lv, d_min, d_max, c.sms, st)) return rc;
    if (E) {
        if (!indexed)                                       // (d_sorted is c.sorted on every path that reaches here)
            if (int e = index_edges(c, d_sorted, N, d_ea, d_eb, E, d_ea, d_eb, st)) return e;
        if (int rc = cluster_mark(d_ea, d_eb, E, d_lv, d_bad, c.sms, st)) return rc;
        if (trace) { cudaStreamSynchronize(st); tr1 = now_ms(); }
        for (int r = 1; r <= rounds; r++) {
            if (int rc = cluster_claim(d_ea, d_eb, E, r, d_ci, d_lv, d_min, d_max, c.sms, st)) return rc;
            if (int rc = cluster_resolve(d_ci, d_lv, d_min, d_max, N, r, c.sms, st)) return rc;
        }
    }
    CU_TRY(cudaGetLastError());
    if (trace) { cudaStreamSynchronize(st); tr2 = now_ms(); }
    if (centre_idx) CU_TRY(cudaMemcpyAsync(centre_idx, d_ci, N * 4, cudaMemcpyDeviceToHost, st));
    if (level) CU_TRY(cudaMemcpyAsync(level, d_lv, N, cudaMemcpyDeviceToHost, st));
    unsigned long long has_edge = 0;
    if (n_has_edge) {
        unsigned long long* d_cnt = (unsigned long long*)((char*)c.cl_flags.p + 8);
        CU_TRY(cudaMemsetAsync(d_cnt, 0, 8, st));
        bdg::count_has_edge_kernel<<<nb, 256, 0, st>>>(d_lv, (uint32_t)N, d_cnt);
        g_launches++;
        CU_TRY(cudaMemcpyAsync(&has_edge, d_cnt, 8, cudaMemcpyDeviceToHost, st));
    }
    unsigned int bad = 0;
    CU_TRY(cudaMemcpyAsync(&bad, d_bad, 4, cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaStreamSynchronize(st));
    if (bad) return fail(BDG_ERR_ARG, "an edge end point is not in the barcode array");
    if (n_has_edge) *n_has_edge = (size_t)has_edge;
    if (trace)
        fprintf(stderr, "[bdg] cluster N=%zu E=%zu: (gather +) seed + index %.2f ms, %d rounds %.2f ms, read-back %.2f ms\n", N, E, tr1 - tr0, rounds,
                tr2 - tr1, now_ms() - tr2);
    return BDG_OK;
}

int bdg_cluster_levels(const uint32_t* sorted_unique, size_t N, const uint32_t* ea, const uint32_t* eb, size_t E, const uint32_t* centres,
                       size_t C, int rounds, int32_t* centre_idx, uint8_t* level)
{
    if (N == 0) return BDG_OK;
    if (!sorted_unique || !centre_idx || !level || (E && (!ea || !eb)) || (C && !centres)) return fail(BDG_ERR_ARG, "NULL pointer argument");
    if (N > 0x7FFFFFFFull || rounds < 0 || rounds > 253) return fail(BDG_ERR_ARG, "N must be < 2^31 and 0 <= rounds <= 253");
    if (int rc = check_sorted(sorted_unique, N)) return rc;
    if (int rc = need_ctx()) return rc;
    DevCtx& c = g_ctx[0];
    CU_TRY(cudaSetDevice(c.dev));
    // the edge workspaces of an earlier build are reused for the index arrays: older handles become stale
    if (int e = c.sorted.ensure(N * 4)) return e;
    if (int e = c.ea.ensure(std::max<size_t>(E, 1) * 4)) return e;
    if (int e = c.eb.ensure(std::max<size_t>(E, 1) * 4)) return e;
    c.generation++;
    CU_TRY(cudaMemcpyAsync(c.sorted.p, sorted_unique, N * 4, cudaMemcpyHostToDevice, c.stream));
    CU_TRY(cudaMemcpyAsync(c.ea.p, ea, E * 4, cudaMemcpyHostToDevice, c.stream));
    CU_TRY(cudaMemcpyAsync(c.eb.p, eb, E * 4, cudaMemcpyHostToDevice, c.stream));
    return cluster_on_device(c, (const uint32_t*)c.sorted.p, N, (uint32_t*)c.ea.p, (uint32_t*)c.eb.p, E, centres, C, rounds, centre_idx, level);
}

static int cluster_from_edges(bdg_edges* e, size_t N, const uint32_t* centres, size_t C, int rounds, int32_t* centre_idx, uint8_t* level, size_t* n_has_edge);

int bdg_cluster_levels_from_edges(bdg_edges* e, size_t N, const uint32_t* centres, size_t C, int rounds, int32_t* centre_idx, uint8_t* level)
{
    if (N && (!centre_idx || !level)) return fail(BDG_ERR_ARG, "NULL pointer argument");
    return cluster_from_edges(e, N, centres, C, rounds, centre_idx, level, nullptr);
}

// The same with the result left on the device for bdg_assign_reads32(token, NULL, ...): no per-node array crosses PCIe.
int bdg_cluster_resident(bdg_edges* e, size_t N, const uint32_t* centres, size_t C, int rounds, size_t* n_has_edge)
{
    if (n_has_edge) *n_has_edge = 0;
    if (int rc = cluster_from_edges(e, N, centres, C, rounds, nullptr, nullptr, n_has_edge)) return rc;
    ReadMap& m = g_ctx[0].map;
    if (e->read_map && e->read_map == m.token && N == m.distinct) m.cl_token = m.token;   // the graph of the live read map
    return BDG_OK;
}

static int cluster_from_edges(bdg_edges* e, size_t N, const uint32_t* centres, size_t C, int rounds, int32_t* centre_idx, uint8_t* level, size_t* n_has_edge)
{
    if (!e) return fail(BDG_ERR_ARG, "NULL edge handle");
    if (N == 0) return BDG_OK;
    if (C && !centres) return fail(BDG_ERR_ARG, "NULL pointer argument");
    if (e->ctx.empty()) return fail(BDG_ERR_ARG, "empty edge handle");
    if (N > 0x7FFFFFFFull || rounds < 0 || rounds > 253) return fail(BDG_ERR_ARG, "N must be < 2^31 and 0 <= rounds <= 253");
    if (int rc = check_edges_handle(e)) return rc;
    DevCtx& c = g_ctx[e->ctx[0]];
    if (c.sorted.cap < N * 4) return fail(BDG_ERR_ARG, "N does not match the array the edges were built from");
    CU_TRY(cudaSetDevice(c.dev));
    if (e->ctx.size() > 1) {
        // Multi-device handle: the parts' edge lists are disjoint (SURVEY.md 8e), so the clustering rounds need their plain
        // concatenation.  It is gathered on the first device with peer copies (NVLink; every part's stream was synchronised
        // by the build), into buffers of its own - the handle's edges stay intact on their devices.
        size_t total = 0;
        for (size_t k : e->count) total += k;
        if (int rc = c.gather_a.ensure(std::max<size_t>(total, 1) * 4)) return rc;
        if (int rc = c.gather_b.ensure(std::max<size_t>(total, 1) * 4)) return rc;
        // every device turns its own edges into node indices (its copy of the array, its SMs), then the indices travel
        size_t off = 0;
        for (size_t g = 0; g < e->ctx.size(); g++) {
            DevCtx& src = g_ctx[e->ctx[g]];
            const size_t k = e->count[g];
            if (k == 0) continue;
            if (&src == &c) {
                CU_TRY(cudaSetDevice(c.dev));
                if (int rc = index_edges(c, (const uint32_t*)c.sorted.p, N, (const uint32_t*)c.ea.p, (const uint32_t*)c.eb.p, k, (uint32_t*)c.gather_a.p + off, (uint32_t*)c.gather_b.p + off, c.stream)) return rc;
            } else {
                CU_TRY(cudaSetDevice(src.dev));
                if (int rc = src.gather_a.ensure(k * 4)) return rc;
                if (int rc = src.gather_b.ensure(k * 4)) return rc;
                if (int rc = index_edges(src, (const uint32_t*)src.sorted.p, N, (const uint32_t*)src.ea.p, (const uint32_t*)src.eb.p, k, (uint32_t*)src.gather_a.p, (uint32_t*)src.gather_b.p, src.stream)) return rc;
                CU_TRY(cudaMemcpyPeerAsync((uint32_t*)c.gather_a.p + off, c.dev, src.gather_a.p, src.dev, k * 4, src.stream));
                CU_TRY(cudaMemcpyPeerAsync((uint32_t*)c.gather_b.p + off, c.dev, src.gather_b.p, src.dev, k * 4, src.stream));
            }
            off += k;
        }
        for (size_t g = 0; g < e->ctx.size(); g++) {             // the rounds start when every part has arrived
            DevCtx& src = g_ctx[e->ctx[g]];
            if (&src == &c || e->count[g] == 0) continue;
            CU_TRY(cudaSetDevice(src.dev));
            CU_TRY(cudaStreamSynchronize(src.stream));
        }
        CU_TRY(cudaSetDevice(c.dev));
        return cluster_on_device(c, (const uint32_t*)c.sorted.p, N, (uint32_t*)c.gather_a.p, (uint32_t*)c.gather_b.p, total, centres, C, rounds, centre_idx, level, n_has_edge, true);
    }
    // the handle's edge VALUES are turned into node indices in place: the handle is consumed (stale afterwards)
    c.generation++;
    return cluster_on_device(c, (const uint32_t*)c.sorted.p, N, (uint32_t*)c.ea.p, (uint32_t*)c.eb.p, e->count[0], centres, C, rounds, centre_idx, level, n_has_edge);
}

// ---- the phases of cluster() on caller-owned node arrays (one process per GPU; include/badger_b200.h) ----
static DevCtx* claimed_current(int* rc)
{
    DevCtx* c = ctx_of_current_device();
    *rc = c ? BDG_OK : fail(BDG_ERR_NODEVICE, "the current device was not claimed by bdg_init");
    return c;
}

int bdg_dev_index_edges(const uint32_t* d_sorted, size_t N, const uint32_t* d_ea, const uint32_t* d_eb, size_t E, uint32_t* d_ia, uint32_t* d_ib,
                        void* stream)
{
    if (!d_sorted || (E && (!d_ea || !d_eb || !d_ia || !d_ib))) return fail(BDG_ERR_ARG, "NULL pointer argument");
    if (N == 0 || N > 0x7FFFFFFFull) return fail(BDG_ERR_ARG, "need 0 < N < 2^31");
    int rc = 0;
    DevCtx* c = claimed_current(&rc);
    if (rc) return rc;
    return index_edges(*c, d_sorted, N, d_ea, d_eb, E, d_ia, d_ib, (cudaStream_t)stream);
}

int bdg_dev_cluster_init(const uint32_t* d_sorted, size_t N, const uint32_t* d_centres, size_t C, int32_t* d_centre_idx, uint8_t* d_level,
                         int32_t* d_cmin, int32_t* d_cmax, void* stream)
{
    if (!d_sorted || !d_centre_idx || !d_level || !d_cmin || !d_cmax || (C && !d_centres)) return fail(BDG_ERR_ARG, "NULL pointer argument");
    if (N == 0 || N > 0x7FFFFFFFull || C > 0xFFFFFFFFull) return fail(BDG_ERR_ARG, "need 0 < N < 2^31 and C < 2^32");
    int rc = 0;
    DevCtx* c = claimed_current(&rc);
    if (rc) return rc;
    return cluster_init(d_sorted, N, d_centres, C, d_centre_idx, d_level, d_cmin, d_cmax, c->sms, (cudaStream_t)stream);
}

int bdg_dev_cluster_mark(const uint32_t* d_ia, const uint32_t* d_ib, size_t E, uint8_t* d_level, unsigned int* d_bad, void* stream)
{
    if (E && (!d_ia || !d_ib || !d_level || !d_bad)) return fail(BDG_ERR_ARG, "NULL pointer argument");
    int rc = 0;
    DevCtx* c = claimed_current(&rc);
    if (rc) return rc;
    return cluster_mark(d_ia, d_ib, E, d_level, d_bad, c->sms, (cudaStream_t)stream);
}

int bdg_dev_cluster_claim(const uint32_t* d_ia, const uint32_t* d_ib, size_t E, int round, const int32_t* d_centre_idx, const uint8_t* d_level,
                          int32_t* d_cmin, int32_t* d_cmax, void* stream)
{
    if (E && (!d_ia || !d_ib || !d_centre_idx || !d_level || !d_cmin || !d_cmax)) return fail(BDG_ERR_ARG, "NULL pointer argument");
    if (round < 1 || round > 253) return fail(BDG_ERR_ARG, "round must be in 1..253");
    int rc = 0;
    DevCtx* c = claimed_current(&rc);
    if (rc) return rc;
    return cluster_claim(d_ia, d_ib, E, round, d_centre_idx, d_level, d_cmin, d_cmax, c->sms, (cudaStream_t)stream);
}

int bdg_dev_cluster_resolve(int32_t* d_centre_idx, uint8_t* d_level, int32_t* d_cmin, int32_t* d_cmax, size_t N, int round, void* stream)
{
    if (!d_centre_idx || !d_level || !d_cmin || !d_cmax) return fail(BDG_ERR_ARG, "NULL pointer argument");
    if (N == 0 || N > 0x7FFFFFFFull || round < 1 || round > 253) return fail(BDG_ERR_ARG, "need 0 < N < 2^31 and round in 1..253");
    int rc = 0;
    DevCtx* c = claimed_current(&rc);
    if (rc) return rc;
    return cluster_resolve(d_centre_idx, d_level, d_cmin, d_cmax, N, round, c->sms, (cudaStream_t)stream);
}

int bdg_member_sorted(const uint32_t* sorted_wl, size_t W, const uint32_t* q, size_t Q, uint8_t* hit)
{
    if (int rc = member_sorted_args(sorted_wl, W, q, Q, hit)) return done(rc);
    DevCtx* c = nullptr;
    if (int rc = first_ctx(&c)) return rc;
    uint32_t *d_wl = nullptr, *d_q = nullptr;
    uint8_t* d_hit = nullptr;
    if (int e = stage(*c, {piece(d_wl, std::max<size_t>(W, 1) * 4), piece(d_q, Q * 4), piece(d_hit, Q)})) return e;
    CU_TRY(cudaMemcpyAsync(d_wl, sorted_wl, W * 4, cudaMemcpyHostToDevice, c->stream));
    CU_TRY(cudaMemcpyAsync(d_q, q, Q * 4, cudaMemcpyHostToDevice, c->stream));
    if (int rc = sort_check(*c, d_wl, W)) return rc;        // the whitelist must be sorted: checked on the device, read back with the hits
    if (int rc = member_sorted_body(d_wl, W, d_q, Q, d_hit, c->stream)) return rc;
    CU_TRY(cudaMemcpyAsync(hit, d_hit, Q, cudaMemcpyDeviceToHost, c->stream));
    return sort_check_result(*c);
}

// The check bdg_member_sorted makes on its whitelist, for a whitelist in device memory (bdg_dev_member_sorted does not check).
int bdg_dev_whitelist_check(const uint32_t* d_sorted_wl, size_t W, void* stream)
{
    if (W <= 1) return BDG_OK;
    if (!d_sorted_wl) return fail(BDG_ERR_ARG, "NULL pointer argument");
    if (W > 0xFFFFFFFFull) return fail(BDG_ERR_ARG, "size exceeds 2^32");
    DevCtx* c = nullptr;
    if (int rc = first_ctx(&c)) return rc;
    if (int rc = check_on_first(d_sorted_wl, "whitelist")) return rc;
    CallerOrder order(*c, stream);
    if (int rc = order.begin()) return rc;
    if (int rc = sort_check(*c, d_sorted_wl, W)) return rc;
    return sort_check_result(*c);
}

int bdg_nearest_bounded(const uint32_t* q, size_t Q, const uint32_t* targets, size_t W, int max_d, int32_t* argmin, uint8_t* dist)
{
    if (Q == 0) return BDG_OK;
    if (!q || !argmin || !dist || (W && !targets)) return fail(BDG_ERR_ARG, "NULL pointer argument");
    if (int rc = need_ctx()) return rc;
    // queries are independent: deal contiguous slices to the devices, targets replicated (SURVEY.md §8e)
    const int G = (int)g_ctx.size();
    int rc = BDG_OK;
    const size_t per = (Q + G - 1) / G;
    for (int g = 0; g < G && rc == BDG_OK; g++) {
        const size_t lo = std::min(Q, per * g), n = std::min(Q, per * (g + 1)) - lo;
        if (n == 0) continue;
        DevCtx& c = g_ctx[g];
        rc = [&]() -> int {
            CU_TRY(cudaSetDevice(c.dev));
            uint32_t *d_q = nullptr, *d_t = nullptr, *d_keys = nullptr;
            int32_t* d_arg = nullptr;
            uint8_t* d_dist = nullptr;
            if (int e = stage(c, {piece(d_q, n * 4), piece(d_t, std::max<size_t>(W, 1) * 4), piece(d_keys, n * 4), piece(d_arg, n * 4),
                                  piece(d_dist, n)})) return e;
            CU_TRY(cudaMemcpyAsync(d_q, q + lo, n * 4, cudaMemcpyHostToDevice, c.stream));
            CU_TRY(cudaMemcpyAsync(d_t, targets, W * 4, cudaMemcpyHostToDevice, c.stream));
            if (int e = bdg_dev_nearest_bounded(d_q, n, d_t, W, max_d, d_keys, d_arg, d_dist, c.stream)) return e;
            CU_TRY(cudaMemcpyAsync(argmin + lo, d_arg, n * 4, cudaMemcpyDeviceToHost, c.stream));
            CU_TRY(cudaMemcpyAsync(dist + lo, d_dist, n, cudaMemcpyDeviceToHost, c.stream));
            return BDG_OK;
        }();
    }
    for (int g = 0; g < G; g++) {
        if (per * g >= Q) continue;
        DevCtx& c = g_ctx[g];
        cudaSetDevice(c.dev);
        cudaError_t e = cudaStreamSynchronize(c.stream);
        if (e != cudaSuccess && rc == BDG_OK) rc = fail(BDG_ERR_CUDA, "stream sync failed: %s", cudaGetErrorString(e));
    }
    cudaSetDevice(g_ctx[0].dev);
    return rc;
}

// ---- a-5  KmerIndexer / QGramIndex: the known strings stay on the device between queries ------------------
static int kmer_index_args(const uint32_t* wl, size_t W, bdg_kmer_index** out, DevCtx** c)
{
    if (!out || (W && !wl)) return fail(BDG_ERR_ARG, "NULL pointer argument");
    *out = nullptr;
    if (W > 0xFFFFFFFFull) return fail(BDG_ERR_ARG, "size exceeds 2^32");
    return first_ctx(c);
}

// wl: the W strings in host memory (kind = cudaMemcpyHostToDevice) or in device memory on the first claimed device
// (cudaMemcpyDeviceToDevice, read on that device's stream, which is ordered after the caller's); copied straight into the index.
static int kmer_index_body(DevCtx& c, const uint32_t* wl, size_t W, bool postings, cudaMemcpyKind kind, cudaStream_t caller, bdg_kmer_index** out)
{
    CallerOrder order(c, caller);
    if (int rc = order.begin()) return rc;
    bdg_kmer_index* ix = new (std::nothrow) bdg_kmer_index();
    if (!ix) return fail(BDG_ERR_OOM, "host allocation failed");
    ix->dev = c.dev;
    ix->W = W;
    if (int e = ix->wl.ensure(std::max<size_t>(W, 1) * 4)) {
        delete ix;
        return e;
    }
    cudaError_t e = cudaMemcpyAsync(ix->wl.p, wl, W * 4, kind, c.stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c.stream);
    if (e != cudaSuccess) { bdg_kmer_index_free(ix); return fail(BDG_ERR_CUDA, "upload of the index failed: %s", cudaGetErrorString(e)); }
    // posting lists of the strings' 6-mers (kmer_indexer.py:29-32): worth it once a bucket is a small share of the strings
    size_t min_w = 4096;
    if (const char* v = getenv("BDG_KMER_POST_MIN_W")) min_w = (size_t)std::max(0ll, atoll(v));
    if (postings && W >= min_w && W > 0 && W <= 0xFFFFFFFFull / 11) {          // (the postings are counted in 32 bits)
        cudaStream_t st = c.stream;
        const int sms = c.sms;
        size_t tmp = 0;
        bool ok = ix->kstart.ensure(4097 * 4) == BDG_OK && ix->scratch.ensure(2 * 4097 * 4) == BDG_OK;
        ok = ok && cub::DeviceScan::ExclusiveSum(nullptr, tmp, (const uint32_t*)nullptr, (uint32_t*)nullptr, 4097, st) == cudaSuccess;
        Buf cubtmp;
        ok = ok && cubtmp.ensure(tmp) == BDG_OK;
        if (ok) {
            uint32_t* hist = (uint32_t*)ix->scratch.p;
            uint32_t* fill = hist + 4097;
            const int nb = (int)std::min<size_t>((W + 255) / 256, (size_t)sms * 8);
            ok = cudaMemsetAsync(hist, 0, 2 * 4097 * 4, st) == cudaSuccess;
            bdg::kidx_hist_kernel<<<nb, 256, 0, st>>>((const uint32_t*)ix->wl.p, (uint32_t)W, hist);
            ok = ok && cub::DeviceScan::ExclusiveSum(cubtmp.p, tmp, (const uint32_t*)hist, (uint32_t*)ix->kstart.p, 4097, st) == cudaSuccess;
            uint32_t n_post = 0;
            ok = ok && cudaMemcpyAsync(&n_post, (uint32_t*)ix->kstart.p + 4096, 4, cudaMemcpyDeviceToHost, st) == cudaSuccess;
            ok = ok && cudaStreamSynchronize(st) == cudaSuccess;
            ok = ok && ix->post.ensure(std::max<size_t>(n_post, 1) * 4) == BDG_OK;
            if (ok) {
                bdg::kidx_scatter_kernel<<<nb, 256, 0, st>>>((const uint32_t*)ix->wl.p, (uint32_t)W, (const uint32_t*)ix->kstart.p, fill, (uint32_t*)ix->post.p);
                g_launches += 2;
                ok = cudaStreamSynchronize(st) == cudaSuccess && cudaGetLastError() == cudaSuccess;
            }
        }
        if (!ok) { bdg_kmer_index_free(ix); return fail(BDG_ERR_CUDA, "building the 6-mer posting lists failed: %s", cudaGetErrorString(cudaGetLastError())); }
        ix->posted = true;
    }
    if (cudaEventCreate(&ix->ev[0]) != cudaSuccess || cudaEventCreate(&ix->ev[1]) != cudaSuccess) {
        bdg_kmer_index_free(ix);
        return fail(BDG_ERR_CUDA, "event creation failed");
    }
    *out = ix;
    return BDG_OK;
}

int bdg_kmer_index_create(const uint32_t* wl, size_t W, bdg_kmer_index** out)
{
    DevCtx* c = nullptr;
    if (int rc = kmer_index_args(wl, W, out, &c)) return rc;
    return kmer_index_body(*c, wl, W, true, cudaMemcpyHostToDevice, c->stream, out);
}

int bdg_dev_kmer_index_create(const uint32_t* d_known, size_t W, void* stream, bdg_kmer_index** out)
{
    DevCtx* c = nullptr;
    if (int rc = kmer_index_args(d_known, W, out, &c)) return rc;
    if (W) if (int rc = check_on_first(d_known, "known")) return rc;
    return kmer_index_body(*c, d_known, W, true, cudaMemcpyDeviceToDevice, (cudaStream_t)stream, out);
}

int bdg_kmer_index_info(const bdg_kmer_index* ix, int* posted, double* kernel_ms)
{
    if (!ix) return fail(BDG_ERR_ARG, "NULL index handle");
    if (posted) *posted = ix->posted ? 1 : 0;
    if (kernel_ms) {
        float ms = 0.f;
        if (ix->timed) CU_TRY(cudaEventElapsedTime(&ms, ix->ev[0], ix->ev[1]));
        *kernel_ms = ms;
    }
    return BDG_OK;
}

void bdg_kmer_index_free(bdg_kmer_index* ix)
{
    if (!ix) return;
    cudaSetDevice(ix->dev);                         // the buffers are freed on their device
    for (auto& e : ix->ev) if (e) cudaEventDestroy(e);
    delete ix;
}

// The query proper, on c (the context of the index's device): d_q (Q queries) on that device, hits appended to d_hq / d_hw / d_cnt
// / d_mult, of which only the first cap are stored.  Waits once, for *tot (the number of hits, which may exceed cap).
static int kmer_query_core(bdg_kmer_index* ix, DevCtx& c, const uint32_t* d_q, size_t Q, int min_kmers, size_t cap, uint32_t* d_hq,
                           uint32_t* d_hw, uint8_t* d_cnt, unsigned long long* d_mult, unsigned long long* tot)
{
    const size_t W = ix->W;
    if (int e = ix->total.ensure(8)) return e;
    unsigned long long* d_total = (unsigned long long*)ix->total.p;
    CU_TRY(cudaMemsetAsync(d_total, 0, 8, c.stream));
    CU_TRY(cudaEventRecord(ix->ev[0], c.stream));
    if (ix->posted) {                                       // walk the buckets of the queries' own 6-mers
        const unsigned blocks = (unsigned)std::min<unsigned long long>((unsigned long long)Q * 11, (unsigned long long)c.sms * 64);
        bdg::kmer_post_kernel<<<blocks, bdg::NT, 0, c.stream>>>(d_q, (uint32_t)Q, (const uint32_t*)ix->wl.p, (const uint32_t*)ix->kstart.p,
                                                              (const uint32_t*)ix->post.p, std::max(min_kmers, 1), (unsigned long long)cap, d_hq, d_hw,
                                                              d_cnt, d_mult, d_total);
    } else {
        const uint32_t gy_total = (uint32_t)((Q + bdg::KS_QB - 1) / bdg::KS_QB);
        const uint32_t gx = (uint32_t)((W + bdg::NT - 1) / bdg::NT);
        if (gy_total > 65535u) return fail(BDG_ERR_ARG, "Q too large for one call (> 65535*256 queries)");
        bdg::kmer_score_kernel<<<dim3(gx, gy_total), bdg::NT, 0, c.stream>>>(d_q, (uint32_t)Q, (const uint32_t*)ix->wl.p, (uint32_t)W, min_kmers,
                                                                          (unsigned long long)cap, d_hq, d_hw, d_cnt, d_mult, d_total);
    }
    g_launches++;
    CU_TRY(cudaGetLastError());
    CU_TRY(cudaEventRecord(ix->ev[1], c.stream));
    ix->timed = true;
    *tot = 0;
    CU_TRY(cudaMemcpyAsync(tot, d_total, 8, cudaMemcpyDeviceToHost, c.stream));
    CU_TRY(cudaStreamSynchronize(c.stream));
    return BDG_OK;
}

int bdg_kmer_index_query(bdg_kmer_index* ix, const uint32_t* q, size_t Q, int min_kmers, size_t cap, uint32_t* hit_q, uint32_t* hit_w,
                         uint8_t* cnt, uint64_t* mult, size_t* total)
{
    if (!total) return fail(BDG_ERR_ARG, "NULL total pointer");
    *total = 0;
    if (!ix) return fail(BDG_ERR_ARG, "NULL index handle");
    if (Q == 0 || ix->W == 0) return BDG_OK;
    if (!q || (cap && (!hit_q || !hit_w || !cnt || !mult))) return fail(BDG_ERR_ARG, "NULL pointer argument");
    if (Q > 0xFFFFFFFFull) return fail(BDG_ERR_ARG, "size exceeds 2^32");
    DevCtx* c = nullptr;
    for (auto& x : g_ctx) if (x.dev == ix->dev) c = &x;
    if (!c) return fail(BDG_ERR_NODEVICE, "the device the index lives on is no longer claimed (bdg_shutdown?)");
    CU_TRY(cudaSetDevice(c->dev));
    const size_t capa = std::max<size_t>(cap, 1);
    for (Buf* b : {&ix->hit_q, &ix->hit_w}) if (int e = b->ensure(capa * 4)) return e;
    if (int e = ix->hit_cnt.ensure(capa)) return e;
    if (int e = ix->mult.ensure(capa * 8)) return e;
    uint32_t* d_q = nullptr;
    if (int e = stage(*c, {piece(d_q, Q * 4)})) return e;
    uint32_t *d_hq = (uint32_t*)ix->hit_q.p, *d_hw = (uint32_t*)ix->hit_w.p;
    uint8_t* d_cnt = (uint8_t*)ix->hit_cnt.p;
    unsigned long long* d_mult = (unsigned long long*)ix->mult.p;
    CU_TRY(cudaMemcpyAsync(d_q, q, Q * 4, cudaMemcpyHostToDevice, c->stream));
    unsigned long long tot = 0;
    if (int rc = kmer_query_core(ix, *c, d_q, Q, min_kmers, cap, d_hq, d_hw, d_cnt, d_mult, &tot)) return rc;
    const size_t n = (size_t)std::min<unsigned long long>(tot, cap);
    if (n) {
        CU_TRY(cudaMemcpyAsync(hit_q, d_hq, n * 4, cudaMemcpyDeviceToHost, c->stream));
        CU_TRY(cudaMemcpyAsync(hit_w, d_hw, n * 4, cudaMemcpyDeviceToHost, c->stream));
        CU_TRY(cudaMemcpyAsync(cnt, d_cnt, n, cudaMemcpyDeviceToHost, c->stream));
        CU_TRY(cudaMemcpyAsync(mult, d_mult, n * 8, cudaMemcpyDeviceToHost, c->stream));
        CU_TRY(cudaStreamSynchronize(c->stream));
    }
    *total = (size_t)tot;
    if (tot > cap) return fail(BDG_ERR_CAPACITY, "%llu hits but room for %zu", tot, cap);
    return BDG_OK;
}

int bdg_dev_kmer_index_query(bdg_kmer_index* ix, const uint32_t* d_q, size_t Q, int min_kmers, size_t cap, uint32_t* d_hit_q, uint32_t* d_hit_w,
                             uint8_t* d_cnt, uint8_t* d_pos, size_t* total, void* stream)
{
    if (!total) return fail(BDG_ERR_ARG, "NULL total pointer");
    *total = 0;
    if (!ix) return fail(BDG_ERR_ARG, "NULL index handle");
    if (Q == 0 || ix->W == 0) return BDG_OK;
    if (!d_q || (cap && (!d_hit_q || !d_hit_w || !d_cnt || !d_pos))) return fail(BDG_ERR_ARG, "NULL pointer argument");
    if (Q > 0xFFFFFFFFull) return fail(BDG_ERR_ARG, "size exceeds 2^32");
    if (g_ctx.empty() || g_ctx[0].dev != ix->dev)
        return fail(BDG_ERR_ARG, "the index lives on device %d, which is not the first claimed device", ix->dev);
    DevCtx& c = g_ctx[0];
    CU_TRY(cudaSetDevice(c.dev));
    if (int rc = check_on_first(d_q, "queries")) return rc;
    if (cap) {
        const void* outs[4] = {d_hit_q, d_hit_w, d_cnt, d_pos};
        for (const void* p : outs) if (int rc = check_on_first(p, "output")) return rc;
    }
    // the position counts are unpacked from library scratch into d_pos; the other outputs are written by the kernels in place
    if (int e = ix->mult.ensure(std::max<size_t>(cap, 1) * 8)) return e;
    unsigned long long* d_mult = (unsigned long long*)ix->mult.p;
    CallerOrder order(c, stream);
    if (int rc = order.begin()) return rc;
    unsigned long long tot = 0;
    if (int rc = kmer_query_core(ix, c, d_q, Q, min_kmers, cap, d_hit_q, d_hit_w, d_cnt, d_mult, &tot)) return rc;
    *total = (size_t)tot;
    if (tot > cap) return fail(BDG_ERR_CAPACITY, "%llu hits but room for %zu", tot, cap);
    if (tot) {
        const unsigned blocks = (unsigned)std::min<unsigned long long>((tot * 11 + 255) / 256, (unsigned long long)c.sms * 16);
        bdg::kmer_unpack_kernel<<<blocks, 256, 0, c.stream>>>(d_mult, tot, d_pos);
        g_launches++;
        CU_TRY(cudaGetLastError());
    }
    return BDG_OK;
}

int bdg_kmer_score(const uint32_t* q, size_t Q, const uint32_t* wl, size_t W, int min_kmers, size_t cap, uint32_t* hit_q,
                   uint32_t* hit_w, uint8_t* cnt, uint64_t* mult, size_t* total)
{
    if (!total) return fail(BDG_ERR_ARG, "NULL total pointer");
    *total = 0;
    if (Q == 0 || W == 0) return BDG_OK;
    if (!q || !wl || (cap && (!hit_q || !hit_w || !cnt || !mult))) return fail(BDG_ERR_ARG, "NULL pointer argument");
    bdg_kmer_index* ix = nullptr;
    DevCtx* c = nullptr;
    if (int rc = kmer_index_args(wl, W, &ix, &c)) return rc;
    if (int rc = kmer_index_body(*c, wl, W, Q >= 64, cudaMemcpyHostToDevice, c->stream, &ix)) return rc;   // a one-off call with few queries: the scan costs less than the lists
    const int rc = bdg_kmer_index_query(ix, q, Q, min_kmers, cap, hit_q, hit_w, cnt, mult, total);
    bdg_kmer_index_free(ix);
    return rc;
}

int bdg_dev_kmer_score(const uint32_t* d_q, size_t Q, const uint32_t* d_wl, size_t W, int min_kmers, size_t cap, uint32_t* d_hit_q,
                       uint32_t* d_hit_w, uint8_t* d_cnt, uint8_t* d_pos, size_t* total, void* stream)
{
    if (!total) return fail(BDG_ERR_ARG, "NULL total pointer");
    *total = 0;
    if (Q == 0 || W == 0) return BDG_OK;
    if (!d_q || !d_wl) return fail(BDG_ERR_ARG, "NULL pointer argument");
    bdg_kmer_index* ix = nullptr;
    DevCtx* c = nullptr;
    if (int rc = kmer_index_args(d_wl, W, &ix, &c)) return rc;
    if (int rc = check_on_first(d_wl, "wl")) return rc;
    if (int rc = kmer_index_body(*c, d_wl, W, Q >= 64, cudaMemcpyDeviceToDevice, (cudaStream_t)stream, &ix)) return rc;   // the rule of bdg_kmer_score
    const int rc = bdg_dev_kmer_index_query(ix, d_q, Q, min_kmers, cap, d_hit_q, d_hit_w, d_cnt, d_pos, total, stream);
    bdg_kmer_index_free(ix);          // cudaFree waits for the unpack kernel that still reads the index's scratch
    return rc;
}

// ---- f-2 / f-4  extraction TSV in, assignment TSV out, whitelist file (host only; bdg_tsv.hpp) -----------------
struct bdg_tsv { tsvio::Tsv t; };
struct bdg_lines16 { tsvio::Lines16 l; };

int bdg_tsv_open(const char* path, int bc_len, int threads, bdg_tsv** out)
{
    if (!path || !out) return fail(BDG_ERR_ARG, "NULL pointer argument");
    *out = nullptr;
    bdg_tsv* h = new (std::nothrow) bdg_tsv();
    if (!h) return fail(BDG_ERR_OOM, "out of host memory");
    bool io = false;
    std::string why;
    try {
        why = tsvio::tsv_parse(h->t, path, bc_len, threads, &io);
    } catch (const std::bad_alloc&) {
        delete h;
        return fail(BDG_ERR_OOM, "out of host memory while reading %s", path);
    }
    if (!why.empty()) {
        delete h;
        return fail(io ? BDG_ERR_IO : BDG_ERR_UNSUPPORTED, "%s%s", io ? "" : "native TSV reader refuses the file: ", why.c_str());
    }
    *out = h;
    return BDG_OK;
}

size_t bdg_tsv_rows(const bdg_tsv* t) { return t ? t->t.rows : 0; }

int bdg_tsv_barcodes(const bdg_tsv* t, char* seqs16, uint8_t* kind)
{
    if (!t) return fail(BDG_ERR_ARG, "NULL TSV handle");
    if (t->t.rows && (!seqs16 || !kind)) return fail(BDG_ERR_ARG, "NULL pointer argument");
    if (t->t.rows) {
        memcpy(seqs16, t->t.seqs.data(), t->t.rows * 16);
        memcpy(kind, t->t.kind.data(), t->t.rows);
    }
    return BDG_OK;
}

int bdg_tsv_write_assignments(const bdg_tsv* t, const char* out_path, const uint64_t* centre_per_row, int threads)
{
    if (!t || !out_path) return fail(BDG_ERR_ARG, "NULL pointer argument");
    if (t->t.rows && !centre_per_row) return fail(BDG_ERR_ARG, "NULL pointer argument");
    std::string why;
    try {
        why = tsvio::tsv_write(t->t, out_path, centre_per_row, threads);
    } catch (const std::bad_alloc&) {
        return fail(BDG_ERR_OOM, "out of host memory while writing %s", out_path);
    }
    if (!why.empty()) return fail(BDG_ERR_IO, "%s", why.c_str());
    return BDG_OK;
}

int bdg_tsv_write_assignments32(const bdg_tsv* t, const char* out_path, const uint32_t* centre_per_row, const uint8_t* has_centre, int threads)
{
    if (!t || !out_path) return fail(BDG_ERR_ARG, "NULL pointer argument");
    if (t->t.rows && (!centre_per_row || !has_centre)) return fail(BDG_ERR_ARG, "NULL pointer argument");
    std::string why;
    try {
        why = tsvio::tsv_write(t->t, out_path, nullptr, threads, centre_per_row, has_centre);
    } catch (const std::bad_alloc&) {
        return fail(BDG_ERR_OOM, "out of host memory while writing %s", out_path);
    }
    if (!why.empty()) return fail(BDG_ERR_IO, "%s", why.c_str());
    return BDG_OK;
}

void bdg_tsv_close(bdg_tsv* t) { delete t; }

int bdg_lines16_open(const char* path, bdg_lines16** out)
{
    if (!path || !out) return fail(BDG_ERR_ARG, "NULL pointer argument");
    *out = nullptr;
    bdg_lines16* h = new (std::nothrow) bdg_lines16();
    if (!h) return fail(BDG_ERR_OOM, "out of host memory");
    bool io = false;
    std::string why;
    try {
        why = tsvio::lines16_read(h->l, path, &io);
    } catch (const std::bad_alloc&) {
        delete h;
        return fail(BDG_ERR_OOM, "out of host memory while reading %s", path);
    }
    if (!why.empty()) {
        delete h;
        return fail(BDG_ERR_IO, "%s", why.c_str());
    }
    *out = h;
    return BDG_OK;
}

size_t bdg_lines16_count(const bdg_lines16* l) { return l ? l->l.count : 0; }
const char* bdg_lines16_data(const bdg_lines16* l) { return l ? l->l.seqs.data() : nullptr; }
void bdg_lines16_close(bdg_lines16* l) { delete l; }

}  // extern "C"
