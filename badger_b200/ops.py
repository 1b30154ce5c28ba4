"""numpy-level operators over the C ABI (host buffers in, host buffers out).

Each function names the reference code it stands in for (file:line in algbio/Badger).
"""
from __future__ import annotations

import ctypes as C
import os
import weakref

import numpy as np

from . import _lib
from .common import sorted_unique  # noqa: F401  (re-exported)
from ._lib import check, lib, ptr

BC_LEN = 16


def pack16(seqs) -> tuple[np.ndarray, np.ndarray]:
    """common.py:21-25 `rank` for many 16-mers at once.  seqs: list of str/bytes (each exactly 16 long), one bytes object
    of R*16 characters, or a uint8 array of R*16 characters.  Returns (ranks uint32[R], valid bool[R])."""
    if isinstance(seqs, np.ndarray):                         # uint8[R, 16] (badger_b200.tsvio records): no copy
        arr = np.ascontiguousarray(seqs, dtype=np.uint8)
        if arr.size % BC_LEN:
            raise ValueError("pack16 needs records of exactly 16 characters")
        R = arr.size // BC_LEN
        out = np.empty(R, np.uint32)
        valid = np.empty(R, np.uint8)
        if R:
            check(lib().bdg_pack16(ptr(arr), R, ptr(out), ptr(valid)))
        return out, valid.astype(bool)
    if isinstance(seqs, (bytes, bytearray, memoryview)):
        buf = bytes(seqs)
    else:
        buf = "".join(seqs).encode("ascii", "replace") if (len(seqs) and isinstance(seqs[0], str)) else b"".join(seqs)
    if len(buf) % BC_LEN:
        raise ValueError("pack16 needs records of exactly 16 characters")
    R = len(buf) // BC_LEN
    out = np.empty(R, np.uint32)
    valid = np.empty(R, np.uint8)
    if R:
        check(lib().bdg_pack16(buf, R, ptr(out), ptr(valid)))
    return out, valid.astype(bool)


def dedup_first_seen(ranks: np.ndarray, want_map: bool = False, want_sorted_pos: bool = False):
    """barcode_graph.py:192-204: distinct barcodes in first-seen order with their counts
    (with want_map also the position in that order of every read; with want_sorted_pos also the position of every
    distinct barcode in ascending order)."""
    r = np.ascontiguousarray(ranks, dtype=np.uint32)
    distinct = np.empty(r.size, np.uint32)
    counts = np.empty(r.size, np.uint32)
    rmap = np.empty(r.size, np.uint32) if want_map else None
    spos = np.empty(r.size, np.uint32) if want_sorted_pos else None
    n = C.c_size_t(0)
    if r.size:
        check(lib().bdg_dedup_first_seen(ptr(r), r.size, ptr(distinct), ptr(counts), ptr(rmap) if want_map else None,
                                         ptr(spos) if want_sorted_pos else None, C.byref(n)))
    k = int(n.value)
    out = (distinct[:k].copy(), counts[:k].astype(np.int64))
    if want_map:
        out += (rmap,)
    if want_sorted_pos:
        out += (spos[:k].copy(),)
    return out


class ReadMap:
    """Result of dedup_reads.  The distinct barcodes (first-seen order), their counts, their ascending positions, the
    ascending array and the read -> barcode map all stay on the device under `token` until the next dedup call; the four
    arrays are downloaded when first asked for (`.distinct`, `.counts`, `.sorted_pos`, `.sorted_distinct`)."""

    def __init__(self, n_distinct, n_valid, rows, token):
        self.n_distinct, self.n_valid, self.rows, self.token = n_distinct, n_valid, rows, token
        self._got = {}

    def _fetch(self, name):
        if name not in self._got:
            n = self.n_distinct
            arr = np.empty(n, np.uint32)
            if n:
                args = [ptr(arr) if k == name else None for k in ("distinct", "counts", "sorted_pos", "sorted_distinct")]
                check(lib().bdg_dedup_fetch(self.token, *args))
            self._got[name] = arr.astype(np.int64) if name == "counts" else arr
        return self._got[name]

    distinct = property(lambda self: self._fetch("distinct"))
    counts = property(lambda self: self._fetch("counts"))
    sorted_pos = property(lambda self: self._fetch("sorted_pos"))
    sorted_distinct = property(lambda self: self._fetch("sorted_distinct"))


def _mask(valid, n):
    """A validity mask for n rows as uint8 for the C ABI (a bool mask is used in place), or None."""
    if valid is None:
        return None
    v = np.ascontiguousarray(valid)
    if v.size != n:
        raise ValueError("valid has %d rows, ranks %d" % (v.size, n))
    return v.view(np.uint8) if v.dtype == np.bool_ else (v != 0).view(np.uint8)


def dedup_reads(ranks: np.ndarray, valid=None) -> ReadMap:
    """barcode_graph.py:192-204 over the rows with valid[i] (None: all), compacted on the device; everything it produces is
    kept there for edges_handle_resident / centres_above / assign_reads (include/badger_b200.h bdg_dedup_reads)."""
    r = np.ascontiguousarray(ranks, dtype=np.uint32)
    v = _mask(valid, r.size)
    n, nv, tok = C.c_size_t(0), C.c_size_t(0), C.c_ulonglong(0)
    if r.size:
        check(lib().bdg_dedup_reads(ptr(r), ptr(v) if v is not None else None, r.size, None, None, None, None,
                                    C.byref(n), C.byref(nv), C.byref(tok)))
    return ReadMap(int(n.value), int(nv.value), int(r.size), int(tok.value))


def centres_above(rmap: ReadMap, n_cells: int, whitelist_sorted=None):
    """barcode_graph.py:252-258 + 264 on the device: (cutoff, top ranks, their counts, whitelist hits or None) - the barcodes
    with count > cutoff in the order of the reference's `bc_by_counts` (count descending, ties by first sighting)."""
    wl = None if whitelist_sorted is None else np.ascontiguousarray(whitelist_sorted, dtype=np.uint32)
    cap = 1 << 16
    while True:
        top = np.empty(cap, np.uint32); cnt = np.empty(cap, np.uint32)
        hits = np.empty(cap, np.uint8) if wl is not None else None
        n, cut = C.c_size_t(0), C.c_double(0.0)
        rc = lib().bdg_centres_above(rmap.token, int(n_cells), ptr(wl) if wl is not None else None, 0 if wl is None else wl.size, ptr(top), ptr(cnt),
                                     ptr(hits) if hits is not None else None, cap, C.byref(n), C.byref(cut))
        if rc == _lib.BDG_ERR_CAPACITY:
            cap = int(n.value)
            continue
        check(rc)
        k = int(n.value)
        return float(cut.value), top[:k], cnt[:k].astype(np.int64), (hits[:k].astype(bool) if hits is not None else None)


def centres_rest(rmap: ReadMap, cutoff: float, need: int) -> np.ndarray:
    """The `need` barcodes that follow the head of centres_above in `bc_by_counts` (count <= cutoff, count-descending, ties by
    first sighting): what the top-up loop of barcode_graph.py:273-276 walks into."""
    need = int(min(max(need, 0), rmap.n_distinct))
    out = np.empty(need, np.uint32)
    n = C.c_size_t(0)
    if need:
        check(lib().bdg_centres_rest(rmap.token, float(cutoff), need, ptr(out), C.byref(n)))
    return out[:int(n.value)].copy()


def pack16_sorted(records) -> np.ndarray:
    """badger.py:82-88 for the array pipeline: uint8[R, 16] records -> ascending distinct packed barcodes (records with letters
    outside ACGT dropped), packed / sorted / made distinct on the device."""
    arr = np.ascontiguousarray(records, dtype=np.uint8)
    if arr.size % BC_LEN:
        raise ValueError("pack16 needs records of exactly 16 characters")
    R = arr.size // BC_LEN
    out = np.empty(R, np.uint32)
    n = C.c_size_t(0)
    if R:
        check(lib().bdg_pack16_sorted(ptr(arr), R, ptr(out), C.byref(n)))
    return out[:int(n.value)].copy()


NONE = np.uint64(1) << np.uint64(32)      # "no centre" in a uint64 per-read result (every uint32 is a valid barcode)


def widen(centre, has_centre) -> np.ndarray:
    """A 5-byte per-read result (assign_reads32) as one uint64 per row: the centre barcode, or NONE where has_centre is 0."""
    out = centre.astype(np.uint64)
    out[has_centre == 0] = NONE
    return out


def assign_reads(rmap: ReadMap, centre_idx: np.ndarray):
    """barcode_graph.py:322-329 + 395-404 on the device: centre barcode of every input row of the dedup call (uint64, 2^32 =
    none) from the clustering result on node positions; returns (centre_per_row, rows with a centre).  assign_reads32, widened."""
    centre, has, n = assign_reads32(rmap, np.ascontiguousarray(centre_idx, dtype=np.int32))
    return widen(centre, has), n


def assign_reads32(rmap: ReadMap, centre_idx=None):
    """assign_reads with a 5-byte result per row: (centre uint32[R], has_centre bool-as-uint8[R], rows with a centre).
    centre_idx None: the clustering EdgeHandle.cluster_resident left on the device is used in place."""
    if rmap.rows and rmap.token:
        out = _pinned.array(rmap.rows, np.uint32)            # page-locked (pooled: allocated by the first call of a size, ~0.4 ms per MB
        has = _pinned.array(rmap.rows, np.uint8)              # once): the per-row result comes back at PCIe speed
    else:
        out = np.zeros(rmap.rows, np.uint32)
        has = np.zeros(rmap.rows, np.uint8)
    n = C.c_size_t(0)
    if rmap.rows and rmap.token:
        ci = None if centre_idx is None else np.ascontiguousarray(centre_idx, dtype=np.int32)
        check(lib().bdg_assign_reads32(rmap.token, ptr(ci) if ci is not None else None, rmap.n_distinct if ci is None else ci.size, ptr(out), ptr(has),
                                       out.size, C.byref(n)))
    return out, has, int(n.value)


class _PinnedPool:
    """Page-locked blocks behind the (large) edge arrays the operators return: a device-to-host copy into pinned memory
    runs at full PCIe speed, into pageable memory at about a third of it.  A block goes back to the pool when the last
    numpy view of it dies; the pool keeps at most POOL_BYTES and frees the rest."""
    POOL_BYTES = int(os.environ.get("BDG_PINNED_POOL_BYTES", str(4 << 30)))
    MIN_BYTES = 1 << 16          # smaller arrays are plain numpy allocations

    def __init__(self):
        self.free = []           # (capacity, address)
        self.held = 0
        self.wanted = set()      # size classes a lazy caller asked for once already

    def take(self, nbytes):
        best = None
        for k, (cap, _) in enumerate(self.free):
            if cap >= nbytes and (best is None or cap < self.free[best][0]) and cap <= 4 * max(nbytes, 1):
                best = k
        if best is not None:
            cap, addr = self.free.pop(best)
            self.held -= cap
            return cap, addr
        cap = (nbytes + (1 << 20) - 1) >> 20 << 20
        p = C.c_void_p()
        check(lib().bdg_host_alloc(cap, C.byref(p)))
        return cap, p.value

    def give(self, cap, addr):
        if _lib._lib is None:
            return
        if self.held + cap <= self.POOL_BYTES:
            self.free.append((cap, addr)); self.held += cap
        else:
            lib().bdg_host_free(addr)

    def array(self, n, dtype, eager=True):
        """eager=False: page-locked memory is only taken from the pool, or allocated when a block of this size class was wanted
        before (cudaHostAlloc costs ~0.4 ms per MB: it pays for a loop over batches, not for a single call)."""
        dtype = np.dtype(dtype)
        nbytes = int(n) * dtype.itemsize
        if nbytes < self.MIN_BYTES:
            return np.empty(n, dtype)
        if not eager:
            size_class = nbytes.bit_length()
            fits = any(cap >= nbytes and cap <= 4 * nbytes for cap, _ in self.free)
            if not fits and size_class not in self.wanted:
                self.wanted.add(size_class)
                return np.empty(n, dtype)
        cap, addr = self.take(nbytes)
        buf = (C.c_char * nbytes).from_address(addr)
        arr = np.frombuffer(buf, dtype=dtype, count=n)        # writable: the ctypes buffer is; views keep `arr` alive through .base
        weakref.finalize(buf, self.give, cap, addr)
        return arr


_pinned = _PinnedPool()


def _collect_edges(handle):
    L = lib()
    try:
        n = L.bdg_edges_count(handle)
        a = _pinned.array(n, np.uint32); b = _pinned.array(n, np.uint32); d = _pinned.array(n, np.uint8)
        check(L.bdg_edges_copy(handle, ptr(a), ptr(b), ptr(d)))
    finally:
        L.bdg_edges_free(handle)
    return a, b, d


class EdgeHandle:
    """Edges of one construction, still on the device (include/badger_b200.h bdg_edges)."""

    def __init__(self, handle, n_nodes):
        self._h, self.n_nodes = handle, n_nodes
        self.count = int(lib().bdg_edges_count(handle))

    def copy(self):
        a = np.empty(self.count, np.uint32); b = np.empty(self.count, np.uint32); d = np.empty(self.count, np.uint8)
        check(lib().bdg_edges_copy(self._h, ptr(a), ptr(b), ptr(d)))
        return a, b, d

    def cluster_levels(self, centres: np.ndarray, rounds: int = 2, want_has_edge: bool = False):
        """barcode_graph.py:279-301 straight from the device-resident edge list; CONSUMES the edges.
        want_has_edge: also return the mask of the non-centre nodes with at least one edge (see ops.cluster_levels)."""
        cen = np.ascontiguousarray(centres, dtype=np.uint32)
        ci = np.full(self.n_nodes, -2, np.int32); lv = np.full(self.n_nodes, 255, np.uint8)
        if self.n_nodes:
            check(lib().bdg_cluster_levels_from_edges(self._h, self.n_nodes, ptr(cen), cen.size, int(rounds), ptr(ci), ptr(lv)))
        return _split_levels(ci, lv, want_has_edge)

    def cluster_resident(self, centres: np.ndarray, rounds: int = 2) -> int:
        """cluster_levels with the result left on the device for assign_reads32(rmap, None); CONSUMES the edges.  Returns the
        number of non-centre nodes with at least one edge."""
        cen = np.ascontiguousarray(centres, dtype=np.uint32)
        n = C.c_size_t(0)
        if self.n_nodes:
            check(lib().bdg_cluster_resident(self._h, self.n_nodes, ptr(cen), cen.size, int(rounds), C.byref(n)))
        return int(n.value)

    def free(self):
        if self._h is not None:
            lib().bdg_edges_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def edges_handle(sorted_unique: np.ndarray, t: int) -> EdgeHandle:
    """Edge construction over all initialised GPUs (rows dealt to them, SURVEY.md 8e), every part left on its device;
    EdgeHandle.cluster_levels gathers the parts on the first device over NVLink."""
    s = np.ascontiguousarray(sorted_unique, dtype=np.uint32)
    h = C.c_void_p()
    check(lib().bdg_edges_build(ptr(s), s.size, int(t), C.byref(h)))
    return EdgeHandle(h, s.size)


def edges_handle_resident(rmap: "ReadMap", t: int) -> EdgeHandle:
    """edges_handle over the ascending distinct barcodes the dedup_reads call left on the first device (no upload)."""
    h = C.c_void_p()
    check(lib().bdg_edges_build_resident(rmap.token, int(t), C.byref(h)))
    return EdgeHandle(h, int(rmap.n_distinct))


def edges_build(sorted_unique: np.ndarray, t: int):
    """index.py:77-93 + barcode_graph.py:224-249 over all initialised GPUs.
    Returns (a, b, d): every undirected edge once with a < b; order unspecified."""
    s = np.ascontiguousarray(sorted_unique, dtype=np.uint32)
    h = C.c_void_p()
    check(lib().bdg_edges_build(ptr(s), s.size, int(t), C.byref(h)))
    return _collect_edges(h)


_cap_hint = {}            # (N, t, nparts) -> edges found last time: the first guess of the next call on the same shape


def edges_build_part(sorted_unique: np.ndarray, t: int, part: int, nparts: int):
    """One part's edges (one process per GPU) straight into page-locked arrays (bdg_edges_build_into): with the join form
    the device-to-host copy runs while later seed conditions are still being joined."""
    s = np.ascontiguousarray(sorted_unique, dtype=np.uint32)
    key = (int(s.size), int(t), int(nparts))
    cap = max(1 << 16, _cap_hint.get(key, ((16 if t <= 1 else 40) * s.size) // max(nparts, 1)) + 1024)
    while True:
        a = _pinned.array(cap, np.uint32); b = _pinned.array(cap, np.uint32); d = _pinned.array(cap, np.uint8)
        n = C.c_size_t(0)
        check(lib().bdg_edges_build_into(ptr(s), s.size, int(t), int(part), int(nparts), ptr(a), ptr(b), ptr(d), cap, C.byref(n)))
        k = int(n.value)
        if k <= cap:
            _cap_hint[key] = k + k // 16
            return a[:k], b[:k], d[:k]
        cap = k + k // 16 + 1024


LEVEL_NONE, LEVEL_HAS_EDGE = 255, 254


def _split_levels(ci, lv, want_has_edge):
    """The library marks nodes no round reached (and evicted ones) that have an edge with level 254; callers of the
    (centre_idx, level) pair see the plain 255 = none."""
    marked = lv == LEVEL_HAS_EDGE
    has_edge = marked | ((lv != LEVEL_NONE) & (lv != 0)) if want_has_edge else None     # joined nodes were reached over an edge
    lv[marked] = LEVEL_NONE
    return (ci, lv, has_edge) if want_has_edge else (ci, lv)


def cluster_levels(sorted_unique: np.ndarray, ea: np.ndarray, eb: np.ndarray, centres: np.ndarray, rounds: int = 2,
                   want_has_edge: bool = False):
    """barcode_graph.py:279-301 on node positions of the sorted array: (centre_idx int32[N], level uint8[N]);
    centre_idx -2 = untouched, -1 = evicted by a same-round conflict, level 255 = none.
    want_has_edge adds the mask of the non-centre nodes with >= 1 edge (centre nodes, level 0, are never marked: the
    reference touches `edges[centre]` whether or not the centre has an edge, barcode_graph.py:293)."""
    s = np.ascontiguousarray(sorted_unique, dtype=np.uint32)
    ea = np.ascontiguousarray(ea, dtype=np.uint32); eb = np.ascontiguousarray(eb, dtype=np.uint32)
    cen = np.ascontiguousarray(centres, dtype=np.uint32)
    ci = np.full(s.size, -2, np.int32)
    lv = np.full(s.size, 255, np.uint8)
    if s.size:
        check(lib().bdg_cluster_levels(ptr(s), s.size, ptr(ea), ptr(eb), ea.size, ptr(cen), cen.size, int(rounds), ptr(ci), ptr(lv)))
    return _split_levels(ci, lv, want_has_edge)


def canonical(a, b, d):
    """Sort an edge list by (a, b) - the order-free comparison form."""
    order = np.lexsort((b, a))
    return a[order], b[order], d[order]


def member_sorted(sorted_wl: np.ndarray, q: np.ndarray) -> np.ndarray:
    """barcode_graph.py:262-267 `unrank(r) in barcode_list` for many r at once."""
    wl = np.ascontiguousarray(sorted_wl, dtype=np.uint32)
    q = np.ascontiguousarray(q, dtype=np.uint32)
    hit = np.zeros(q.size, np.uint8)
    if q.size:
        check(lib().bdg_member_sorted(ptr(wl), wl.size, ptr(q), q.size, ptr(hit)))
    return hit.astype(bool)


def nearest_bounded(q: np.ndarray, targets_in_order: np.ndarray, max_d: int = 2):
    """barcode_graph.py:370-385: first minimum of the plain edit distance over the targets, kept if <= max_d."""
    q = np.ascontiguousarray(q, dtype=np.uint32)
    tg = np.ascontiguousarray(targets_in_order, dtype=np.uint32)
    am = np.full(q.size, -1, np.int32)
    dist = np.full(q.size, 255, np.uint8)
    if q.size:
        check(lib().bdg_nearest_bounded(ptr(q), q.size, ptr(tg), tg.size, int(max_d), ptr(am), ptr(dist)))
    return am, dist


def _kmer_query(call, q, n_known, min_kmers, cap, hint=None):
    """hint: a one-element list that carries the room the last call needed to the next one (a resident index is queried many
    times with similar batches; a first guess that is too small costs one repeated launch with the exact size)."""
    q = np.ascontiguousarray(q, dtype=np.uint32)
    if cap is None:
        cap = hint[0] if hint and hint[0] else max(1 << 16, min(4 * n_known, 2048 * max(int(q.size), 1)))
    while True:
        hq = np.empty(cap, np.uint32); hw = np.empty(cap, np.uint32)
        cnt = np.empty(cap, np.uint8); mult = np.empty(cap, np.uint64)
        total = C.c_size_t(0)
        rc = call(ptr(q), q.size, int(min_kmers), cap, ptr(hq), ptr(hw), ptr(cnt), ptr(mult), C.byref(total))
        if rc == _lib.BDG_ERR_CAPACITY:
            cap = int(total.value) + int(total.value) // 8
            continue
        check(rc)
        n = int(total.value)
        if hint is not None:
            hint[0] = max(1 << 16, n + n // 8)
        by = mult[:n].view(np.uint8).reshape(n, 8)          # little-endian: nibble p of the word = nibble p & 1 of byte p >> 1
        nib = np.empty((n, 16), np.uint8)
        np.bitwise_and(by, 15, out=nib[:, 0::2])
        np.right_shift(by, 4, out=nib[:, 1::2])
        return hq[:n].copy(), hw[:n].copy(), cnt[:n].copy(), nib[:, :11]


def kmer_score(q: np.ndarray, wl: np.ndarray, min_kmers: int = 1, cap: int | None = None):
    """kmer_indexer.py:49-61 counting step for packed 16-mers, k=6.
    Returns (hit_q, hit_w, cnt, mult[hits,11]) for every pair with cnt >= min_kmers (order unspecified)."""
    wl = np.ascontiguousarray(wl, dtype=np.uint32)
    L = lib()
    return _kmer_query(lambda *a: L.bdg_kmer_score(a[0], a[1], ptr(wl), wl.size, *a[2:]), q, wl.size, min_kmers, cap)


class KmerIndex:
    """The known strings of a KmerIndexer / QGramIndex, uploaded once and kept on the device (bdg_kmer_index)."""

    def __init__(self, known: np.ndarray):
        known = np.ascontiguousarray(known, dtype=np.uint32)
        self.size = int(known.size)
        self._h = C.c_void_p()
        check(lib().bdg_kmer_index_create(ptr(known), known.size, C.byref(self._h)))
        self._room = [0]

    def query(self, q: np.ndarray, min_kmers: int = 1, cap: int | None = None):
        L = lib()
        return _kmer_query(lambda *a: L.bdg_kmer_index_query(self._h, *a), q, self.size, min_kmers, cap, self._room)

    def info(self) -> dict:
        """{"postings": queries walk 6-mer posting lists (else they scan every string), "kernel_ms": the last query's kernel}."""
        posted, ms = C.c_int(0), C.c_double(0.0)
        check(lib().bdg_kmer_index_info(self._h, C.byref(posted), C.byref(ms)))
        return {"postings": bool(posted.value), "kernel_ms": float(ms.value)}

    def free(self):
        if self._h is not None and self._h.value:
            lib().bdg_kmer_index_free(self._h)
        self._h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass
