/*
 * badger_b200.h -- C ABI of libbadger_b200.so: the B200-native replacement for the barcode
 * edit-distance hot path of algbio/Badger.
 *
 * The reference is pure Python and has no FFI of its own; the seam this library sits behind is the set
 * of Python methods listed beside each entry point (file:line in the reference checkout).  The Python
 * package badger_b200/ binds these symbols with ctypes and mirrors those methods; INTEGRATION.md shows
 * the stub a maintainer of the reference would add.
 *
 * Conventions
 *   - plain pointers and sizes only; host entry points take HOST buffers (read-only during the call) and
 *     do their own host<->device copies; bdg_dev_* entry points take DEVICE pointers on the current CUDA
 *     device plus a cudaStream_t passed as void*, and are asynchronous on that stream (the correction-step ones
 *     take pointers on the first claimed device and order their work against that stream; see below).
 *   - every int-returning function returns BDG_OK (0) or a negative error code; bdg_last_error() gives the
 *     text.  There is NO CPU fallback: without a usable CUDA device every compute call fails with
 *     BDG_ERR_NODEVICE.
 *   - barcodes are uint32 in the reference's packing (common.py:21-25): base i in bits 2i..2i+1, A0 C1 G2 T3.
 *   - the library is not re-entrant across threads except bdg_last_error (thread-local).
 */
#ifndef BADGER_B200_H
#define BADGER_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

enum {
    BDG_OK = 0,
    BDG_ERR_CUDA = -1,     /* a CUDA runtime call failed */
    BDG_ERR_OOM = -2,      /* host or device allocation failed */
    BDG_ERR_ARG = -3,      /* bad argument (NULL, unsorted input, size limit) */
    BDG_ERR_NODEVICE = -4, /* no CUDA device / library not initialised on one */
    BDG_ERR_CAPACITY = -5, /* caller-provided output capacity too small; *total holds the need */
    BDG_ERR_UNSUPPORTED = -6, /* bdg_tsv_open: the file uses a construct the native reader refuses (take the pandas route);
                                 bdg_join_lane_stats: the build does not count */
    BDG_ERR_IO = -7        /* a file could not be opened, mapped or written */
};

/* How the edge construction is dealt to parts (GPUs / ranks); the parts' edge lists are disjoint and their union is the full edge
 * set, so they are simply concatenated (no exchange step).  Replaces the 10 000-barcode chunks dealt to worker processes in
 * barcode_graph.py:26,164-189.
 *   join form (t = 2, 3): the seed conditions are laid on a line by estimated work and the line is cut into nparts equal pieces; a
 *     part buckets and joins only the conditions its piece touches, a condition on a cut is shared by row range, cut at a bucket
 *     boundary (the same on every part, because it depends on the bucket sizes only);
 *   sparse / dense forms: rows of the (rotated) sort order in tiles of BDG_ROW_TILE rows, boustrophedon: tile I belongs to part
 *     m<P ? m : 2P-1-m,  m = I mod 2P (dense: a part emits every edge whose SMALLER barcode lies in one of its tiles). */
#define BDG_ROW_TILE 2048

/* ---- life cycle ------------------------------------------------------------------------------- */
/* Create per-device contexts (stream, scratch).  device_ids == NULL or n_devices <= 0: every visible
 * device.  Idempotent for the same list.  Replaces ProcessPoolExecutor(max_workers=threads)
 * (barcode_graph.py:142,177). */
int bdg_init(const int* device_ids, int n_devices);
void bdg_shutdown(void);
int bdg_device_count(void);         /* devices held by this process after bdg_init, else 0 */
const char* bdg_last_error(void);   /* thread-local; valid until the next call on this thread */
const char* bdg_version(void);

/* Page-locked host memory (cudaHostAlloc) for output buffers: device-to-host copies into it run at full PCIe speed. */
int bdg_host_alloc(size_t bytes, void** out);
void bdg_host_free(void* p);

/* ---- a-1  rank(): common.py:21-25 (called per read at barcode_graph.py:198) ----------------------- */
/* seqs: R records of exactly 16 bytes, no terminator.  valid[i] = 1 iff all 16 bytes are in "ACGT"
 * (the reference raises KeyError otherwise, common.py:24); out[i] is undefined when valid[i] == 0. */
int bdg_pack16(const char* seqs, size_t R, uint32_t* out, uint8_t* valid);
/* The whitelist file's records (badger.py:82-88) for the array pipeline: packed, records with other letters dropped, sorted,
 * made distinct - all on the device.  out_sorted has room for R entries; *n receives the number kept. */
int bdg_pack16_sorted(const char* seqs, size_t R, uint32_t* out_sorted, size_t* n);

/* ---- a-2  index_bc_single_thread: barcode_graph.py:192-204 ------------------------------------------ */
/* Dedup + count of R packed barcodes in read order (already length-filtered and valid).  distinct[] receives the
 * distinct barcodes in the order of their FIRST sighting (the iteration order of the reference's `counts` dict),
 * counts[] their multiplicities, read_to_distinct[] (optional, may be NULL) the position in distinct[] of every read,
 * sorted_pos[] (optional) the position each distinct barcode has in ASCENDING order (so the sorted array the edge
 * construction wants is sorted[sorted_pos[p]] = distinct[p]).  Outputs are caller-allocated with room for R entries;
 * *n_distinct receives the number of distinct barcodes. */
int bdg_dedup_first_seen(const uint32_t* ranks, size_t R, uint32_t* distinct, uint32_t* counts, uint32_t* read_to_distinct,
                         uint32_t* sorted_pos, size_t* n_distinct);

/* ---- f-1 / f-2 with the per-read arrays resident on the device -------------------------------------------------- */
/* bdg_dedup_reads = bdg_dedup_first_seen over the rows with valid[i] != 0 (valid == NULL: all rows), compacted on the
 * device; the read -> barcode map is NOT copied out but kept on the first device, and *token names it.
 * bdg_assign_reads32 is the per-read half of assign_by_cluster + output_file (barcode_graph.py:322-329, 395-404), and the
 * library's only per-read gather: centre_idx[N] is the clustering result on node positions of the ascending array
 * (bdg_cluster_levels*, possibly patched by the caller, e.g. for --high_sens); for every input row of the dedup call,
 * centre_per_row[R_all] receives the barcode of the centre its barcode was assigned to and has_centre[R_all] 1, or both 0
 * (rows with valid == 0, unassigned / evicted barcodes: the reference writes '*').  *n_assigned = rows with a centre.
 * centre_idx == NULL: the clustering result a bdg_cluster_resident call left on the device is used in place - no per-node
 * array crosses PCIe in either direction.  The token dies with the next dedup call.  (A caller that wants one uint64 per row,
 * 2^32 for "no centre", widens this result on the host, as badger_b200.ops.widen does.) */
int bdg_dedup_reads(const uint32_t* ranks, const uint8_t* valid, size_t R_all, uint32_t* distinct, uint32_t* counts,
                    uint32_t* sorted_pos, uint32_t* sorted_distinct /* optional: the distinct barcodes ascending */,
                    size_t* n_distinct, size_t* n_valid, unsigned long long* token);
int bdg_assign_reads32(unsigned long long token, const int32_t* centre_idx, size_t N, uint32_t* centre_per_row, uint8_t* has_centre,
                       size_t R_all, size_t* n_assigned);
/* bdg_dedup_reads accepts NULL for distinct / counts / sorted_pos / sorted_distinct (nothing is downloaded then);
 * bdg_dedup_fetch downloads any of them later, while the token is alive. */
int bdg_dedup_fetch(unsigned long long token, uint32_t* distinct, uint32_t* counts, uint32_t* sorted_pos, uint32_t* sorted_distinct);

/* ---- a-6 + centre selection: barcode_graph.py:252-267 over the distinct barcodes of a bdg_dedup_reads call ---------------- */
/* *cutoff = max(mean(counts of the first n_cells barcodes in first-seen order) / 5, 5) (:255-256).  top_ranks / top_counts
 * (room for cap entries) receive the barcodes with count > cutoff in count-descending order, ties in first-seen order: the head
 * of the reference's `bc_by_counts` (:253).  top_hits (optional) receives `unrank(r) in barcode_list` (:264) for each of them,
 * looked up in sorted_wl[W] on the device.  *n_above = their number; BDG_ERR_CAPACITY when it exceeds cap.  The walk over
 * that head (:262-277) is a few thousand steps and stays with the caller. */
int bdg_centres_above(unsigned long long token, size_t n_cells, const uint32_t* sorted_wl, size_t W, uint32_t* top_ranks,
                      uint32_t* top_counts, uint8_t* top_hits, size_t cap, size_t* n_above, double* cutoff);
/* The stretch of `bc_by_counts` right behind that head, for the top-up loop of barcode_graph.py:273-276: the first `need`
 * barcodes with count <= floor(cutoff), count-descending, ties in first-seen order (out_ranks has room for `need`). */
int bdg_centres_rest(unsigned long long token, double cutoff, size_t need, uint32_t* out_ranks, size_t* n_out);

/* ---- a-3 + a-4  QGramIndex.get_close + verify/emit: index.py:77-93, barcode_graph.py:224-249 ------ */
/* Edge set {(a,b,D): a<b, S(a,b) >= T(t), D(a,b) <= t} over a STRICTLY INCREASING array of distinct
 * barcodes (checked).  bdg_edges_build uses every initialised device (rows dealt per BDG_ROW_TILE) and
 * returns the union; bdg_edges_build_part computes one part on the first initialised device (one process
 * per GPU).  Edge order is unspecified.  t <= 0 yields the empty set, as in the reference. */
/* The handle keeps the edges in device memory until bdg_edges_copy moves them straight into the caller's arrays; it
 * becomes stale (BDG_ERR_ARG from bdg_edges_copy) once another edge build runs on the same device - copy first. */
typedef struct bdg_edges bdg_edges;
int bdg_edges_build(const uint32_t* sorted_unique, size_t N, int t, bdg_edges** out);
int bdg_edges_build_part(const uint32_t* sorted_unique, size_t N, int t, int part, int nparts, bdg_edges** out);
/* The same over the ascending distinct barcodes that the bdg_dedup_reads call named by `token` left on the first device: no
 * upload; with several devices the array fans out over NVLink peer copies. */
int bdg_edges_build_resident(unsigned long long token, int t, bdg_edges** out);
/* One part's edges straight into caller buffers of cap entries each (page-locked buffers - bdg_host_alloc - copy at PCIe
 * speed).  With the join form the finished edges of earlier seed conditions cross PCIe while later conditions are still being
 * joined, so the copy hides behind the kernels.  *count = edges found; if it exceeds cap only the first cap were stored: repeat
 * the call with more room (the edge set is deterministic). */
int bdg_edges_build_into(const uint32_t* sorted_unique, size_t N, int t, int part, int nparts, uint32_t* a, uint32_t* b, uint8_t* d,
                         size_t cap, size_t* count);
size_t bdg_edges_count(const bdg_edges* e);
int bdg_edges_copy(const bdg_edges* e, uint32_t* a, uint32_t* b, uint8_t* d); /* caller-allocated, length = count */
void bdg_edges_free(bdg_edges* e);

/* ---- f-3  cluster(): barcode_graph.py:279-301 (the two level-synchronous rounds with same-round conflict eviction) -- */
/* Nodes are positions in sorted_unique[N].  centres[C]: barcode values of the cluster centres (values that are not in
 * sorted_unique are ignored: a centre that was never observed has no node).  On return centre_idx[i] = position of the
 * centre node i joined, -1 if two centres claimed it in the same round (the reference's (-1,-1)), -2 if no round reached
 * it; level[i] = 0 for centres, the round number for joined nodes, 254 for nodes no round reached that have at least one
 * edge (what `len(graph.edges.keys())`, badger.py:131, needs), 255 otherwise.  The reference runs rounds = 2 (<= 253).
 * bdg_cluster_levels takes the edge list from host arrays (barcode values, each undirected edge once);
 * bdg_cluster_levels_from_edges takes it from an edge handle without a trip through the host (N = the size of the array
 * the handle was built from).  A single-device handle is used in place and CONSUMED: copy its edges out first if they are
 * still needed.  The parts of a multi-device handle (bdg_edges_build on several GPUs) are gathered on the handle's first
 * device with peer copies over NVLink - the only inter-GPU transfer of the whole path - and stay intact. */
int bdg_cluster_levels(const uint32_t* sorted_unique, size_t N, const uint32_t* ea, const uint32_t* eb, size_t E,
                       const uint32_t* centres, size_t C, int rounds, int32_t* centre_idx, uint8_t* level);
int bdg_cluster_levels_from_edges(bdg_edges* e, size_t N, const uint32_t* centres, size_t C, int rounds, int32_t* centre_idx,
                                  uint8_t* level);
/* The same with the result left on the first device for bdg_assign_reads32(token, NULL, ...).  *n_has_edge = nodes that are no
 * centre and have at least one edge (what `len(graph.edges.keys())`, badger.py:131, counts beside the centres).  The result
 * belongs to the read map the handle was built from (bdg_edges_build_resident), and only while that read map's token is live. */
int bdg_cluster_resident(bdg_edges* e, size_t N, const uint32_t* centres, size_t C, int rounds, size_t* n_has_edge);

/* ---- a-6  whitelist membership: `unrank(r) in barcode_list`, barcode_graph.py:262-267 -------------- */
int bdg_member_sorted(const uint32_t* sorted_wl, size_t W, const uint32_t* q, size_t Q, uint8_t* hit);

/* ---- a-7  postprocessing(): barcode_graph.py:370-385 ---------------------------------------------- */
/* For every q: the FIRST index (in the given order) of the minimum plain edit distance to the targets,
 * kept when that minimum is <= max_d (the reference's `min_dist < 3` is max_d = 2); else argmin = -1,
 * dist = 255.  W < 2^28. */
int bdg_nearest_bounded(const uint32_t* q, size_t Q, const uint32_t* targets_in_order, size_t W, int max_d,
                        int32_t* argmin, uint8_t* dist);

/* ---- a-5  KmerIndexer.get_occurrences counting step: kmer_indexer.py:49-61 (k = 6, 16-mers) -------- */
/* All (query, entry) pairs with cnt = #{(p,p'): 6mer_q[p] == 6mer_wl[p']} >= min_kmers.  mult packs, 4 bits
 * per query position p = 0..10, the number of matching positions of the entry (the reference's
 * `positions` list is p repeated mult[p] times).  Outputs are caller-allocated with room for cap hits;
 * *total receives the number found; BDG_ERR_CAPACITY when total > cap (first cap hits are valid).
 * Also serves QGramIndex.get_close (index.py:77-93): min_kmers = T(t), keep entries > query. */
int bdg_kmer_score(const uint32_t* q, size_t Q, const uint32_t* wl, size_t W, int min_kmers, size_t cap,
                   uint32_t* hit_q, uint32_t* hit_w, uint8_t* cnt, uint64_t* mult, size_t* total);

/* The same with the known strings kept on the device between queries - the life cycle of the reference's index objects
 * (KmerIndexer.__init__ / QGramIndex.add_to_index build once, get_occurrences / get_close query many times). */
typedef struct bdg_kmer_index bdg_kmer_index;
int bdg_kmer_index_create(const uint32_t* wl, size_t W, bdg_kmer_index** out);
int bdg_kmer_index_query(bdg_kmer_index* ix, const uint32_t* q, size_t Q, int min_kmers, size_t cap, uint32_t* hit_q,
                         uint32_t* hit_w, uint8_t* cnt, uint64_t* mult, size_t* total);
void bdg_kmer_index_free(bdg_kmer_index* ix);
/* *posted: 1 when the index holds 6-mer posting lists (from 4096 strings on; BDG_KMER_POST_MIN_W) and queries walk the buckets
 * of their own 6-mers, 0 when every query scans every string.  *kernel_ms: device time of the last query's kernel.  Either may be NULL. */
int bdg_kmer_index_info(const bdg_kmer_index* ix, int* posted, double* kernel_ms);

/* ---- device-resident variants (bench.py "value" path; torch owns the memory and the stream) -------- */
/* Edge construction over rows of part/nparts.  d_count (one uint64, device) is zeroed by the call and receives
 * the number of edges found, which may exceed cap (only the first cap are stored).  The current device must have
 * been claimed by bdg_init (the call uses its workspaces).  Fully asynchronous.  If bit 63 of *d_count is set after
 * the stream has drained, a sparse pass found more candidate tiles than the device's tile list holds (adversarial,
 * extremely dense inputs): call bdg_edges_build_part once (it grows the list) or use dense mode, then repeat. */
int bdg_dev_edges_build(const uint32_t* d_sorted, size_t N, int t, int part, int nparts, uint32_t* d_a,
                        uint32_t* d_b, uint8_t* d_d, size_t cap, unsigned long long* d_count, void* stream);
/* How the edge set is searched (results are identical; DESIGN.md "edge construction"):
 *   2 join (t = 2, 3): sort-merge joins on multi-block seeds - per seed condition the array is sorted by the condition's
 *     key, equal-key buckets are paired and only those pairs are tested (bdg_join.cuh); the default for t = 2
 *     from BDG_JOIN_MIN_N (150 000) distinct barcodes upwards, for t = 3 from BDG_JOIN3_MIN_N (90 000) upwards;
 *   1 sparse (default otherwise): one pass per prefilter block over the array sorted by a rotated key, pairs are decided
 *     tile by tile from key intervals and scored only inside the tiles that can hold a candidate;
 *   0 dense: one pass, the low-block conditions are scored for every pair (the all-pairs kernel);
 *  -1 back to the default / BDG_EDGE_MODE=dense|sparse|join.  t = 3 has no sparse form: modes 0 and 1 run it dense, below
 *     BDG_JOIN3_MIN_N too; t >= 4 always runs dense without a block prefilter. */
int bdg_set_edge_mode(int mode);
/* Work statistics of the last bdg_dev_edges_build / bdg_edges_build* launch on the current device, summed over
 * its passes: out5[0] column sub-tiles whose key interval was tested, out5[1] sub-tiles that could hold a
 * candidate, out5[2] pairs scored pair by pair (sparse: quick test; dense: light loop or full prefilter),
 * out5[3] candidates handed to the exact stage, out5[4] pairs with D <= t whose 6-mer score S was computed (sparse
 * mode only).  Synchronises the stream.  (bench.py's roofline numerator.) */
int bdg_dev_edges_stats(unsigned long long* out5, void* stream);
/* The kernels' eight raw counters of the last edge launch on the current device, summed over its passes.  Join form: [0] work
 * units, [2] pairs tested, [3] candidates handed to the exact stage, [6] candidates with D <= t, [7] of those, the ones this
 * condition owns, whose 6-mer score was computed; [4] / [5] sum / max over the warps of their busy time in ns.  Synchronises the stream. */
int bdg_dev_edges_stats_raw(unsigned long long* out8, void* stream);
/* Development aid: out[2p], out[2p+1] = sum and max over the warps of pass p of (warp exit - first warp start), ns. */
int bdg_dev_edges_balance(unsigned long long* out6, void* stream);
/* Development aid: lane use of the join kernel, summed over its launches on the current device since the last reset (reset != 0
 * clears them after the read): out8[0] push rounds, [1] hits pushed, [2] candidate batches through the exact distance, [3] their
 * candidates, [4] those batches with a pair at D <= t, [5] batches through the hand-over check, [6] their pairs.  Only in a build
 * with -DBDG_JOIN_LANE_STATS; otherwise BDG_ERR_UNSUPPORTED.  Synchronises the device. */
int bdg_join_lane_stats(unsigned long long* out8, int reset);
int bdg_dev_pack16(const char* d_seqs, size_t R, uint32_t* d_out, uint8_t* d_valid, void* stream);
int bdg_dev_member_sorted(const uint32_t* d_sorted_wl, size_t W, const uint32_t* d_q, size_t Q, uint8_t* d_hit,
                          void* stream);

/* ---- the correction step with the per-read arrays in caller device memory ------------------------------------------------
 * Device forms of bdg_dedup_reads / bdg_dedup_fetch / bdg_pack16_sorted / bdg_centres_above / bdg_edges_copy / bdg_assign_reads32:
 * the same kernels and results, but the per-read and per-barcode arrays are read from and written to caller memory on the FIRST
 * device given to bdg_init (where the read map lives); a pointer to any other memory is BDG_ERR_ARG.  The work runs on the
 * library's stream of that device, ordered after everything queued on `stream` before the call, and `stream` is ordered after
 * the work of the call: the inputs may be produced, and the outputs consumed, by kernels on `stream` without a synchronisation.
 * A call synchronises only where its host form does to learn a size (*n_valid / *n_distinct, *n, *n_above, *n_assigned); only
 * such sizes and scalars cross PCIe.  Tokens have the life cycle of the host forms. */
/* bdg_dedup_reads with every output pointer NULL; d_valid may be NULL (all rows valid).  The valid bytes are copied into the
 * library's workspace (the per-read gather reads them again), so the caller's arrays are free once the call returns. */
int bdg_dev_dedup_reads(const uint32_t* d_ranks, const uint8_t* d_valid, size_t R_all, size_t* n_distinct, size_t* n_valid,
                        unsigned long long* token, void* stream);
/* bdg_dedup_fetch into device buffers of n_distinct entries; any pointer may be NULL. */
int bdg_dev_dedup_fetch(unsigned long long token, uint32_t* d_distinct, uint32_t* d_counts, uint32_t* d_sorted_pos,
                        uint32_t* d_sorted_distinct, void* stream);
/* bdg_pack16_sorted over R records of 16 bytes on the device (16-byte aligned); d_out_sorted has room for R entries. */
int bdg_dev_pack16_sorted(const char* d_seqs, size_t R, uint32_t* d_out_sorted, size_t* n, void* stream);
/* bdg_centres_above with the sorted whitelist on the device; top_ranks / top_counts / top_hits stay HOST buffers (the head of a few
 * thousand entries is walked on the host). */
int bdg_dev_centres_above(unsigned long long token, size_t n_cells, const uint32_t* d_sorted_wl, size_t W, uint32_t* top_ranks,
                          uint32_t* top_counts, uint8_t* top_hits, size_t cap, size_t* n_above, double* cutoff, void* stream);
/* bdg_edges_copy into device buffers of bdg_edges_count(e) entries; the parts of a multi-device handle arrive by peer copies. */
int bdg_dev_edges_copy(const bdg_edges* e, uint32_t* d_a, uint32_t* d_b, uint8_t* d_d, void* stream);
/* bdg_assign_reads32 with a device centre_idx (NULL: the clustering bdg_cluster_resident left on the device) and device outputs
 * of R_all rows.  n_assigned may be NULL: the call then does not wait for the gather. */
int bdg_dev_assign_reads32(unsigned long long token, const int32_t* d_centre_idx, size_t N, uint32_t* d_centre_per_row,
                           uint8_t* d_has_centre, size_t R_all, size_t* n_assigned, void* stream);

/* ---- the correction step over P processes, one per GPU (badger_b200.distributed) ------------------------------------------
 * Every process dedups its own reads (bdg_dev_dedup_reads), the processes exchange their distinct lists, and each reduces the
 * P lists to the global distinct set with bdg_dev_dedup_merge.  The reads of part 0 come first, then those of part 1, ...:
 * the global first sighting of a barcode is the smallest (part, local first-seen position).
 * d_keys / d_counts / d_first: device memory on the first claimed device; part p's list has sizes[p] entries at index starts[p]
 * (host arrays of n_parts): its distinct barcodes ASCENDING, their counts, and their local first-seen positions.  The list of
 * my_part must be the one of the read map `token` names (checked: size, and every barcode on the device); token 0 stands for a
 * part without a valid read, whose list is empty.  The parts hold fewer than 2^31 barcodes in all.
 * On success *merged_token names a read map that holds THIS part's reads and the GLOBAL barcodes (N = *n_distinct):
 *   distinct (dd[2])  in global first-seen order          counts (dd[0])  summed over the parts, in that order
 *   sorted_pos (dd[1]) global first-seen -> ascending     sorted_distinct (dd[6]) ascending
 *   the read -> barcode map (dd[7]) points at global first-seen positions; the valid rows are those of the dedup call.
 * bdg_dev_dedup_fetch, bdg_dev_centres_above, bdg_centres_rest and bdg_dev_assign_reads32 (with a device centre_idx over the N
 * global nodes) take the merged token as they take a dedup token; `token` itself dies.  On error the token stays as it was. */
int bdg_dev_dedup_merge(unsigned long long token, const uint32_t* d_keys, const uint32_t* d_counts, const uint32_t* d_first,
                        const size_t* starts, const size_t* sizes, int n_parts, int my_part, size_t* n_distinct,
                        unsigned long long* merged_token, void* stream);

/* ---- the correction step over reads that arrive in batches (a tally) ----------------------------------------------------------
 * add batches 0 .. B-1 in order, finish, then assign any rows: the per-read result equals what the one-call step
 * (bdg_dedup_reads ... bdg_assign_reads32) gives for the concatenation of the batches.  Every batch holds fewer than 2^31 rows;
 * the total may exceed 2^32.
 *   tally_create  a handle on the first claimed device.  It keeps the running distinct set in its own buffers (not in the dedup
 *                 workspace): every distinct barcode ascending, its 64-bit count and its 64-bit first sighting.  tally_free
 *                 releases them.  A handle is refused (BDG_ERR_ARG) once its device is no longer the first claimed one.
 *   tally_add     dedups the batch (the rows with valid[i] != 0; valid == NULL: all) with the dedup kernels and merges its
 *                 ascending distinct list into the set (merge path; counts summed, the smaller first sighting kept).  *n_valid
 *                 (may be NULL) = valid rows of the batch.  Like any dedup call, it kills the read map of an outstanding token.
 *                 BDG_ERR_ARG after finish, for a batch of 2^31 rows or more, and for a batch that would take the set to 2^31
 *                 distinct barcodes or more (the set keeps the batches before it).  Waits for the batch's sizes.
 *   tally_finish  sorts the set by first sighting and installs it as the read map of a dedup call WITHOUT rows (*token; 0 when no
 *                 valid row was added): distinct in first-seen order, counts, sorted_pos and sorted_distinct as bdg_dev_dedup_merge
 *                 documents them, so bdg_edges_build_resident, bdg_[dev_]centres_above, bdg_centres_rest, bdg_cluster_resident and
 *                 bdg_[dev_]dedup_fetch take the token unchanged.  *n_distinct = barcodes, *n_valid = valid rows added in all.  A
 *                 barcode counted 2^32 times or more is refused with BDG_ERR_ARG (the read map's counts are uint32).  The tally
 *                 takes no more batches afterwards; finish may be called again, to install the read map anew after a later
 *                 dedup call killed the token.
 *   assign_lookup32  the per-read gather for rows that are in no read map: every valid row's barcode is looked up among the nodes
 *                 of the read map `token` names (its ascending array), node -> centre node (centre_idx[N] over those nodes; NULL:
 *                 the result bdg_cluster_resident left for this read map) -> centre barcode.  centre / has_centre as for
 *                 bdg_assign_reads32; *n_assigned = rows with a centre, *n_missing = valid rows whose barcode is no node (their
 *                 has_centre is 0).  Any token works, a dedup call's too.  The device form waits only when n_assigned or
 *                 n_missing is given.
 *   tally_info    *n_distinct = barcodes in the running set, *rows / *valid = rows and valid rows added so far.
 * Over P processes (badger_b200.distributed.Tally), every process adds its own batches to its own tally; then the P sets become
 * one.  The merge order is RANK-MAJOR: part 0's batches in add order, then part 1's, ...  The result equals one tally that added
 * that concatenation of batches.
 *   dev_tally_copy  the running set, ascending, into device buffers of tally_info's *n_distinct entries: barcodes, counts and
 *                 first sightings (the rows added before the batch of the first sighting + the barcode's first-seen position in it).
 *   dev_tally_merge_parts  replaces the set with the union of the P parts' sets.  d_keys / d_cnts / d_firsts: device memory on the
 *                 first claimed device; part p's set has sizes[p] entries at index starts[p] of each array (host arrays of n_parts,
 *                 as bdg_dev_tally_copy wrote them), and its first sightings are shifted by row_offsets[p], the rows of the parts
 *                 before it.  Counts are summed, and the smallest shifted first sighting is kept.  *rows / *valid of the handle become
 *                 total_rows / total_valid, so that finish sorts the first sightings of all parts.  The parts are folded into the
 *                 set one by one, part 0 first (a merge path over every entry of the running union per part).  BDG_ERR_ARG, with
 *                 the set as it was, for a part whose barcodes are not strictly ascending or whose shifted first sightings are not
 *                 below total_rows, a part my_part that is not this handle's set (size, and every entry on the device), a union of
 *                 2^31 barcodes or more, a finished handle, and pointers off the first claimed device.  A merged count of 2^32 or
 *                 more is not refused here: tally_finish refuses it, on every part alike.  After the merge the tally takes no
 *                 more batches and no second merge; tally_finish follows.  Waits for the size of every step.
 * The bdg_dev_* forms take pointers on the first claimed device and order their work against `stream` as the correction-step
 * device forms above do. */
typedef struct bdg_tally bdg_tally;
int bdg_tally_create(bdg_tally** out);
void bdg_tally_free(bdg_tally* h);
int bdg_tally_add(bdg_tally* h, const uint32_t* ranks, const uint8_t* valid, size_t R, size_t* n_valid);
int bdg_dev_tally_add(bdg_tally* h, const uint32_t* d_ranks, const uint8_t* d_valid, size_t R, size_t* n_valid, void* stream);
int bdg_tally_finish(bdg_tally* h, size_t* n_distinct, size_t* n_valid, unsigned long long* token);
int bdg_dev_tally_finish(bdg_tally* h, size_t* n_distinct, size_t* n_valid, unsigned long long* token, void* stream);
int bdg_tally_info(bdg_tally* h, size_t* n_distinct, unsigned long long* rows, unsigned long long* valid);
int bdg_dev_tally_copy(bdg_tally* h, uint32_t* d_key, unsigned long long* d_cnt, unsigned long long* d_first, void* stream);
int bdg_dev_tally_merge_parts(bdg_tally* h, const uint32_t* d_keys, const unsigned long long* d_cnts, const unsigned long long* d_firsts,
                              const size_t* starts, const size_t* sizes, const unsigned long long* row_offsets, int n_parts, int my_part,
                              unsigned long long total_rows, unsigned long long total_valid, void* stream);
int bdg_assign_lookup32(unsigned long long token, const int32_t* centre_idx, size_t N, const uint32_t* ranks, const uint8_t* valid, size_t R,
                        uint32_t* centre, uint8_t* has_centre, size_t* n_assigned, size_t* n_missing);
int bdg_dev_assign_lookup32(unsigned long long token, const int32_t* d_centre_idx, size_t N, const uint32_t* d_ranks, const uint8_t* d_valid,
                            size_t R, uint32_t* d_centre, uint8_t* d_has_centre, size_t* n_assigned, size_t* n_missing, void* stream);
/* The phases of bdg_cluster_levels over node arrays the caller owns, on `stream` of the current (claimed) device and without a
 * synchronisation, so that processes can reduce the claims between the phases.  Nodes are positions in d_sorted[N]
 * (0 < N < 2^31); d_centre_idx / d_level as for bdg_cluster_levels, except that level 254 marks a node with an edge that no
 * round reached; d_cmin / d_cmax (int32[N]) hold the claims of the running round.
 *   index_edges  edge end points (barcode values) -> node indices (in place when d_ia == d_ea); an end point that is not a node
 *                turns both ends of its edge into 0xFFFFFFFF, which cluster_mark reports through *d_bad != 0
 *   cluster_init every node free, no claims; the centres (barcode values, d_centres[C]) that are nodes seeded at level 0
 *   cluster_mark level 255 -> 254 at both ends of every edge
 *   cluster_claim (round r = 1, 2, ...)  every edge from a node joined at level r-1 to a free node records its centre in the free
 *                node's min / max: over several edge lists, reduce d_cmin by minimum and d_cmax by maximum before the resolve
 *   cluster_resolve (round r)  a claimed node joins when min == max and is evicted otherwise; clears the claims
 * The reference runs rounds 1 and 2. */
int bdg_dev_index_edges(const uint32_t* d_sorted, size_t N, const uint32_t* d_ea, const uint32_t* d_eb, size_t E, uint32_t* d_ia,
                        uint32_t* d_ib, void* stream);
int bdg_dev_cluster_init(const uint32_t* d_sorted, size_t N, const uint32_t* d_centres, size_t C, int32_t* d_centre_idx,
                         uint8_t* d_level, int32_t* d_cmin, int32_t* d_cmax, void* stream);
int bdg_dev_cluster_mark(const uint32_t* d_ia, const uint32_t* d_ib, size_t E, uint8_t* d_level, unsigned int* d_bad, void* stream);
int bdg_dev_cluster_claim(const uint32_t* d_ia, const uint32_t* d_ib, size_t E, int round, const int32_t* d_centre_idx,
                          const uint8_t* d_level, int32_t* d_cmin, int32_t* d_cmax, void* stream);
int bdg_dev_cluster_resolve(int32_t* d_centre_idx, uint8_t* d_level, int32_t* d_cmin, int32_t* d_cmax, size_t N, int round,
                            void* stream);
int bdg_dev_nearest_bounded(const uint32_t* d_q, size_t Q, const uint32_t* d_targets, size_t W, int max_d,
                            uint32_t* d_keys /* Q words of scratch */, int32_t* d_argmin, uint8_t* d_dist,
                            void* stream);

/* ---- the whitelist operators (a-5, a-6) with the strings and the results in caller device memory --------------------------
 * Pointers on the first claimed device (else BDG_ERR_ARG); the work runs on the library's stream of that device, ordered as the
 * correction-step device forms above.  bdg_dev_member_sorted and bdg_dev_nearest_bounded run on `stream` itself.
 *   whitelist_check  the sortedness check of bdg_member_sorted (BDG_ERR_ARG "whitelist not sorted at index i"); waits for 8 bytes
 *   kmer_index_create  bdg_kmer_index_create from W strings on the device (same posting-list rule, BDG_KMER_POST_MIN_W)
 *   kmer_index_query   bdg_kmer_index_query into device buffers of cap hits: d_hit_q, d_hit_w, d_cnt as there, d_pos as
 *                      uint8[cap][11] (the position counts of query positions 0..10, unpacked).  The index must live on the first
 *                      claimed device.  Waits once, for *total; when *total > cap: BDG_ERR_CAPACITY, d_pos untouched and nothing
 *                      beyond cap entries written.
 *   kmer_score         bdg_kmer_score on the device: a one-off index (posting lists from 64 queries upwards) and one query. */
int bdg_dev_whitelist_check(const uint32_t* d_sorted_wl, size_t W, void* stream);
int bdg_dev_kmer_index_create(const uint32_t* d_known, size_t W, void* stream, bdg_kmer_index** out);
int bdg_dev_kmer_index_query(bdg_kmer_index* ix, const uint32_t* d_q, size_t Q, int min_kmers, size_t cap, uint32_t* d_hit_q,
                             uint32_t* d_hit_w, uint8_t* d_cnt, uint8_t* d_pos, size_t* total, void* stream);
int bdg_dev_kmer_score(const uint32_t* d_q, size_t Q, const uint32_t* d_wl, size_t W, int min_kmers, size_t cap, uint32_t* d_hit_q,
                       uint32_t* d_hit_w, uint8_t* d_cnt, uint8_t* d_pos, size_t* total, void* stream);
/* Number of pairs the edge kernel decides for this part: sum over owned rows i of (N-1-i). */
unsigned long long bdg_part_pairs(size_t N, int part, int nparts);
/* Kernel launches issued by this process so far (bench.py's gpu_launches). */
unsigned long long bdg_launch_count(void);

/* Integer-pipe roofline probe (SURVEY.md §8d: the INT peak is not in MEASURED_PEAKS.json and must be
 * measured).  kind 0: LOP3 only (ALU pipe), 1: IMAD only (FMA pipe), 2: LOP3+IMAD interleaved 1:1,
 * 3: POPC.  Runs `iters` loop trips of 64 independent warp instructions per thread on blocks x 256
 * threads; the caller times it with CUDA events.  *ops_per_thread receives the instruction count. */
int bdg_dev_pipe_probe(int kind, int blocks, int iters, uint32_t* d_sink, unsigned long long* ops_per_thread,
                       void* stream);

/* ---- f-2 / f-4  the files either side of the path (host code, no device needed) --------------------------------
 * bdg_tsv_open reads an extraction TSV the way badger.py:91-111 does through pandas.read_csv(sep="\t"): header line
 * with `#read_id` and `barcode` columns, blank lines skipped, short rows padded with NaN, the NA strings of pandas ->
 * no barcode, repeated header rows dropped, 17-character barcodes cut to 16 (barcode_graph.py:195-196, badger.py:107).
 * Files with anything else pandas would treat specially (quotes, carriage returns, NUL / non-ASCII bytes, rows longer
 * than the header, ids or barcodes that look like numbers / booleans) are refused with BDG_ERR_UNSUPPORTED and must be
 * read through pandas.  Memory-mapped, `threads` parser threads (<= 0: all cores).
 *   rows           data rows of the file (every non-blank line after the header)
 *   barcodes       seqs16[rows*16]: the first 16 characters of the row's barcode ('A' x 16 when it has none);
 *                  kind[rows]: bit 0 = the row's barcode goes into the graph (16/17 characters, not '*', not NaN, not a
 *                  repeated header; LETTERS ARE NOT CHECKED HERE - bdg_pack16 does that on the GPU), bit 1 = the row is
 *                  written to the output (badger.py:103-110)
 *   write          barcode_graph.py:388-410 / to_csv(sep="\t", index=False): `readID\tbarcode`, then per written row its id
 *                  and the unranked centre_per_row[row] (common.py:27-38), or `*` when that value is >= 2^32. */
typedef struct bdg_tsv bdg_tsv;
int bdg_tsv_open(const char* path, int bc_len, int threads, bdg_tsv** out);
size_t bdg_tsv_rows(const bdg_tsv* t);
int bdg_tsv_barcodes(const bdg_tsv* t, char* seqs16, uint8_t* kind);
int bdg_tsv_write_assignments(const bdg_tsv* t, const char* out_path, const uint64_t* centre_per_row, int threads);
int bdg_tsv_write_assignments32(const bdg_tsv* t, const char* out_path, const uint32_t* centre_per_row, const uint8_t* has_centre, int threads);
void bdg_tsv_close(bdg_tsv* t);

/* Whitelist file, badger.py:82-88 (`set(file.read().split("\n"))`): the entries of exactly 16 characters, 16 bytes each
 * (no other entry can equal an unranked barcode, barcode_graph.py:264).  data stays valid until close. */
typedef struct bdg_lines16 bdg_lines16;
int bdg_lines16_open(const char* path, bdg_lines16** out);
size_t bdg_lines16_count(const bdg_lines16* l);
const char* bdg_lines16_data(const bdg_lines16* l);
void bdg_lines16_close(bdg_lines16* l);

#ifdef __cplusplus
}
#endif
#endif /* BADGER_B200_H */
