"""The correction step on CUDA tensors: the operators of ``ops`` and ``pipeline.assign_packed`` for callers whose barcodes are
already on the GPU (a torch pipeline, or letters read into a CUDA tensor and packed with ``pack16``), and the whitelist
operators ``member_sorted``, ``nearest_bounded``, ``kmer_score`` and ``KmerIndex``, whose per-query and per-hit arrays stay there.

Tensors live on the first device given to ``badger_b200.init`` (where the library keeps the read map) and every call runs in
order with ``torch.cuda.current_stream()`` of that device: inputs produced there, and outputs consumed there, need no
synchronisation.  The per-read arrays never cross PCIe; only sizes, scalars and the short head of the count-ordered barcode
list do (and, with ``high_sens``, the per-barcode work of ``pipeline.assign_packed``).

Barcodes are ``torch.int32`` or ``torch.uint32`` tensors holding the uint32 packing of ``common.rank`` (the same bits) and come
back in the dtype they came in; arrays the library makes from letters (``pack16``, ``pack16_sorted``) are ``torch.int32``.
Sorted barcode arrays are ascending as uint32.  Masks are ``torch.bool`` (``torch.uint8`` is accepted: non-zero = true).
"""
from __future__ import annotations

import ctypes as C
import os
import time

import numpy as np
import torch

from . import _lib, ops, pipeline
from ._lib import check, lib

BARCODE_DTYPES = (torch.int32, torch.uint32)
MASK_DTYPES = (torch.bool, torch.uint8)


def _device() -> torch.device:
    return torch.device("cuda", _lib.first_device())


def _stream():
    return C.c_void_p(torch.cuda.current_stream(_device()).cuda_stream)


def _ptr(t):
    return None if t is None or t.numel() == 0 else t.data_ptr()


def _check(t, name, dtypes, ndim=1):
    """Reject what the library cannot take before any call reaches it."""
    if not isinstance(t, torch.Tensor):
        raise TypeError("%s must be a torch.Tensor, not %s" % (name, type(t).__name__))
    if t.dtype not in dtypes:
        raise TypeError("%s has dtype %s; expected %s" % (name, t.dtype, " or ".join(str(d) for d in dtypes)))
    dev = _device()
    if t.device.type != "cuda":
        raise ValueError("%s is on %s; badger_b200.device takes CUDA tensors on %s" % (name, t.device, dev))
    if t.device.index != dev.index:
        raise ValueError("%s is on %s, not on %s (the first device given to badger_b200.init)" % (name, t.device, dev))
    if t.dim() != ndim:
        raise ValueError("%s must have %d dimension(s), not %d" % (name, ndim, t.dim()))
    if not t.is_contiguous():
        raise ValueError("%s must be contiguous" % name)


def _check_records(seqs, name):
    _check(seqs, name, (torch.uint8,), ndim=2)
    if seqs.shape[1] != ops.BC_LEN:
        raise ValueError("%s must be [R, 16] (records of exactly 16 characters), not %s" % (name, list(seqs.shape)))
    if seqs.numel() and seqs.data_ptr() % 16:
        raise ValueError("%s must start on a 16-byte boundary" % name)


def _rows(ranks, valid):
    """Reject barcodes per row, or their validity mask (None: all rows valid), that the library cannot take; returns them."""
    _check(ranks, "ranks", BARCODE_DTYPES)
    if valid is not None:
        _check(valid, "valid", MASK_DTYPES)
        if valid.numel() != ranks.numel():
            raise ValueError("valid has %d rows, ranks %d" % (valid.numel(), ranks.numel()))
    return ranks, valid


def _check_whitelist(whitelist_sorted):
    if whitelist_sorted is not None:
        _check(whitelist_sorted, "whitelist_sorted", BARCODE_DTYPES)
    return whitelist_sorted


def _true_barcodes(true_barcodes):
    """--true_barcodes as pipeline.select_centres takes them: a tensor becomes the list of its uint32 values."""
    if isinstance(true_barcodes, torch.Tensor):
        return (true_barcodes.to(torch.int64) & 0xFFFFFFFF).tolist()
    return true_barcodes


def _zeros(ranks):
    """The result of rows none of which has a centre: (centre[R] in the dtype of ranks, has_centre bool[R]), all zero."""
    R, dev = ranks.numel(), ranks.device
    return torch.zeros(R, dtype=ranks.dtype, device=dev), torch.zeros(R, dtype=torch.bool, device=dev)


def _ready():
    """The library's contexts, claimed the way the host operators claim them when nobody called init()."""
    if lib().bdg_device_count() == 0:
        _lib.init()


def pack16(seqs: torch.Tensor):
    """common.py:21-25 `rank` of R records: uint8[R, 16] letters -> (ranks int32[R], valid bool[R]); ranks[i] is undefined where
    valid[i] is false (a letter outside ACGT)."""
    _ready()
    _check_records(seqs, "seqs")
    R = seqs.shape[0]
    out = torch.empty(R, dtype=torch.int32, device=seqs.device)
    valid = torch.empty(R, dtype=torch.bool, device=seqs.device)
    if R:
        with torch.cuda.device(seqs.device):
            check(lib().bdg_dev_pack16(seqs.data_ptr(), R, out.data_ptr(), valid.data_ptr(), _stream()))
    return out, valid


def pack16_sorted(records: torch.Tensor) -> torch.Tensor:
    """badger.py:82-88 for the array pipeline (ops.pack16_sorted): uint8[R, 16] whitelist records -> the ascending distinct packed
    barcodes (int32 tensor), records with letters outside ACGT dropped."""
    _ready()
    _check_records(records, "records")
    R = records.shape[0]
    out = torch.empty(R, dtype=torch.int32, device=records.device)
    n = C.c_size_t(0)
    if R:
        check(lib().bdg_dev_pack16_sorted(records.data_ptr(), R, out.data_ptr(), C.byref(n), _stream()))
    return out[:int(n.value)]


def _edge_cap(n, t, nparts=1):
    """First guess of the edge buffer size; BDG_EDGE_CAP_PER_ROW overrides the edges per row, as for the host builds."""
    per_row = int(os.environ.get("BDG_EDGE_CAP_PER_ROW", 16 if t <= 1 else 64))
    return max(1 << 16, max(per_row, 1) * n // nparts + 1024)


def edges(sorted_unique: torch.Tensor, t: int, *, part: int = 0, nparts: int = 1):
    """index.py:77-93 + barcode_graph.py:224-249 (ops.edges_build) on the first device: (a, b, d), every undirected edge once with
    a < b, order unspecified; a / b in the dtype of sorted_unique, d uint8.  sorted_unique must be strictly increasing as uint32
    (not checked here; ops.edges_build checks it).  Waits once for the edge count; when the first guess of the buffer size was
    too small, the build runs again with the exact size (the edge set is deterministic).  part / nparts: only the edges of that
    part of the construction (include/badger_b200.h BDG_ROW_TILE); the nparts parts are disjoint and their union is the edge set."""
    _ready()
    _check(sorted_unique, "sorted_unique", BARCODE_DTYPES)
    if not 0 <= part < nparts:
        raise ValueError("part %d of %d parts" % (part, nparts))
    dev, n, L = sorted_unique.device, sorted_unique.numel(), lib()
    count = torch.zeros(1, dtype=torch.int64, device=dev)
    cap = _edge_cap(n, t, nparts)
    with torch.cuda.device(dev):
        for _ in range(2):
            a = torch.empty(cap, dtype=sorted_unique.dtype, device=dev)
            b = torch.empty(cap, dtype=sorted_unique.dtype, device=dev)
            d = torch.empty(cap, dtype=torch.uint8, device=dev)
            check(L.bdg_dev_edges_build(_ptr(sorted_unique), n, int(t), int(part), int(nparts), a.data_ptr(), b.data_ptr(), d.data_ptr(),
                                        cap, count.data_ptr(), _stream()))
            k = int(count.item())
            if k < 0:
                # bit 63: a sparse pass listed more candidate tiles than the device's tile list holds (adversarial, extremely dense
                # inputs).  The host build grows the list and its result is the edge set: copy that one out.
                return _edges_host_build(sorted_unique, t, part, nparts)
            if k <= cap:
                return a[:k], b[:k], d[:k]
            cap = k
    raise _lib.BadgerB200Error(_lib.BDG_ERR_CUDA, "edge construction did not settle after growing its buffers (count %d)" % k)


def _edges_host_build(sorted_unique, t, part, nparts):
    s = sorted_unique.cpu().numpy().view(np.uint32)
    h = C.c_void_p()
    check(lib().bdg_edges_build_part(_lib.ptr(s), s.size, int(t), int(part), int(nparts), C.byref(h)))
    try:
        return edges_copy(h, sorted_unique.dtype)
    finally:
        lib().bdg_edges_free(h)


def edges_copy(handle, dtype=torch.int32):
    """bdg_dev_edges_copy: the edges of a bdg_edges handle (ops.EdgeHandle or its raw pointer) as (a, b, d) tensors on the first
    device; the parts of a handle built on several devices arrive by peer copies."""
    h = handle._h if isinstance(handle, ops.EdgeHandle) else handle
    n = int(lib().bdg_edges_count(h))
    dev = _device()
    a = torch.empty(n, dtype=dtype, device=dev)
    b = torch.empty(n, dtype=dtype, device=dev)
    d = torch.empty(n, dtype=torch.uint8, device=dev)
    check(lib().bdg_dev_edges_copy(h, _ptr(a), _ptr(b), _ptr(d), _stream()))
    return a, b, d


class DeviceReadMap(ops.ReadMap):
    """ops.ReadMap of a dedup_reads call on tensors: the same token and sizes; `.distinct`, `.counts`, `.sorted_pos` and
    `.sorted_distinct` are tensors on the first device, copied there from the library's workspace when first asked for
    (barcodes in the dtype of the input, counts and positions int64).  `.host` is the same read map for the host operators."""

    def __init__(self, n_distinct, n_valid, rows, token, dtype):
        super().__init__(n_distinct, n_valid, rows, token)
        self.dtype = dtype
        self.host = ops.ReadMap(n_distinct, n_valid, rows, token)

    def _fetch(self, name):
        if name not in self._got:
            n = self.n_distinct
            arr = torch.empty(n, dtype=torch.int32 if name in ("counts", "sorted_pos") else self.dtype, device=_device())
            if n:
                args = [arr.data_ptr() if k == name else None for k in ("distinct", "counts", "sorted_pos", "sorted_distinct")]
                check(lib().bdg_dev_dedup_fetch(self.token, *args, _stream()))
            self._got[name] = arr.to(torch.int64) if name in ("counts", "sorted_pos") else arr
        return self._got[name]


def dedup_reads(ranks: torch.Tensor, valid: torch.Tensor | None = None) -> DeviceReadMap:
    """barcode_graph.py:192-204 over the rows with valid[i] (None: all), as ops.dedup_reads: everything it produces stays on the
    device under the token until the next dedup call; the caller's tensors are free again when it returns."""
    _ready()
    _rows(ranks, valid)
    R = ranks.numel()
    n, nv, tok = C.c_size_t(0), C.c_size_t(0), C.c_ulonglong(0)
    if R:
        check(lib().bdg_dev_dedup_reads(ranks.data_ptr(), _ptr(valid), R, C.byref(n), C.byref(nv), C.byref(tok), _stream()))
    return DeviceReadMap(int(n.value), int(nv.value), R, int(tok.value), ranks.dtype)


def centres_above(rmap, n_cells: int, whitelist_sorted: torch.Tensor | None = None):
    """ops.centres_above with the sorted whitelist in a tensor on the first device; the result (a few thousand barcodes) is on
    the host, where walk_centres runs."""
    wl = _check_whitelist(whitelist_sorted)
    cap = 1 << 16
    while True:
        top = np.empty(cap, np.uint32); cnt = np.empty(cap, np.uint32)
        hits = np.empty(cap, np.uint8) if wl is not None else None
        n, cut = C.c_size_t(0), C.c_double(0.0)
        rc = lib().bdg_dev_centres_above(rmap.token, int(n_cells), _ptr(wl), 0 if wl is None else wl.numel(), _lib.ptr(top),
                                         _lib.ptr(cnt), _lib.ptr(hits) if hits is not None else None, cap, C.byref(n), C.byref(cut),
                                         _stream())
        if rc == _lib.BDG_ERR_CAPACITY:
            cap = int(n.value)
            continue
        check(rc)
        k = int(n.value)
        return float(cut.value), top[:k], cnt[:k].astype(np.int64), (hits[:k].astype(bool) if hits is not None else None)


def assign_packed(ranks: torch.Tensor, valid: torch.Tensor | None = None, *, threshold, n_cells, interval=25, whitelist_sorted=None,
                  true_barcodes=None, high_sens=False, centre_order=None, timings=None):
    """pipeline.assign_packed(form="u32") on tensors: ((centre[R] in the dtype of ranks, has_centre bool[R]), info), the same
    stages and the same `info`.  centre[i] is meaningful where has_centre[i]; elsewhere the reference writes ``*``.

    whitelist_sorted: a tensor of ascending barcodes on the first device (e.g. from pack16_sorted) or None; true_barcodes: an
    iterable of packed centres or a tensor; centre_order: as for pipeline.assign_packed.  Without high_sens nothing of size R or
    N crosses PCIe; with high_sens the per-barcode --high_sens work runs on the host as in pipeline.assign_packed, and the
    per-read arrays still stay on the device.  timings: a dict that receives the host time of every stage, as in
    pipeline.assign_packed."""
    _ready()
    _check(ranks, "ranks", BARCODE_DTYPES)
    _check_whitelist(whitelist_sorted)
    true_barcodes = _true_barcodes(true_barcodes)
    T = timings if timings is not None else {}
    R, dev = ranks.numel(), ranks.device
    info = {"reads": int(R)}
    t0 = time.perf_counter()
    rm = dedup_reads(ranks, valid)
    pipeline._tick(T, "dedup_first_seen", t0)
    info["valid_reads"] = int(rm.n_valid)
    if rm.n_valid == 0:
        return _zeros(ranks), info

    def gather(ci):
        # ci: None (the clustering result on the device) or, with high_sens, the patched centre index per node from the host
        d_ci = None if ci is None else torch.from_numpy(np.ascontiguousarray(ci, dtype=np.int32)).to(dev)
        centre = torch.empty(R, dtype=ranks.dtype, device=dev)
        has = torch.empty(R, dtype=torch.bool, device=dev)
        n = C.c_size_t(0)
        check(lib().bdg_dev_assign_reads32(rm.token, _ptr(d_ci), rm.n_distinct, centre.data_ptr(), has.data_ptr(), R, C.byref(n),
                                           _stream()))
        return (centre, has), int(n.value)

    out = pipeline.run_stages(rm.host, info, T, pipeline._OneProcess(), gather, threshold=threshold, n_cells=n_cells, interval=interval,
                              whitelist_sorted=whitelist_sorted, true_barcodes=true_barcodes, high_sens=high_sens,
                              centre_order=centre_order, centres_above=centres_above)
    return out, info


class Tally(pipeline.Tally):
    """pipeline.Tally on tensors: add(ranks, valid=None) and assign(ranks, valid=None) take tensors on the first device (checked
    as dedup_reads checks them); assign returns (centre[R] in the dtype of its ranks, has_centre bool[R]).  finish takes
    whitelist_sorted as a tensor on the first device and true_barcodes as an iterable or a tensor.  Nothing of size R or N
    crosses PCIe in add or assign; with high_sens the patched node -> centre array is uploaded once, by finish."""

    _centres_above = staticmethod(centres_above)
    _rows = staticmethod(_rows)
    _zeros = staticmethod(_zeros)

    def __init__(self):
        _ready()
        super().__init__()

    def add(self, ranks: torch.Tensor, valid: torch.Tensor | None = None) -> int:
        _rows(ranks, valid)
        R = ranks.numel()
        nv = C.c_size_t(0)
        check(lib().bdg_dev_tally_add(self._handle(), _ptr(ranks), _ptr(valid), R, C.byref(nv), _stream()))
        self.rows += R
        return int(nv.value)

    def _close(self, stages, T, args):
        args["true_barcodes"] = _true_barcodes(args["true_barcodes"])
        return super()._close(stages, T, args)

    def _finish_call(self, n, nv, tok):
        check(lib().bdg_dev_tally_finish(self._handle(), C.byref(n), C.byref(nv), C.byref(tok), _stream()))

    def _upload(self, ci):
        return torch.as_tensor(ci, dtype=torch.int32, device=_device())

    def _lookup(self, rm, ranks, valid):
        R, dev = ranks.numel(), ranks.device
        centre = torch.empty(R, dtype=ranks.dtype, device=dev)
        has = torch.empty(R, dtype=torch.bool, device=dev)
        na, nm = C.c_size_t(0), C.c_size_t(0)
        check(lib().bdg_dev_assign_lookup32(rm.token, _ptr(self._ci), rm.n_distinct, _ptr(ranks), _ptr(valid), R, _ptr(centre), _ptr(has),
                                            C.byref(na), C.byref(nm), _stream()))
        return centre, has, int(na.value), int(nm.value)


# ---------------------------------------------------------------------------------------------- the whitelist operators
def member_sorted(sorted_wl: torch.Tensor, q: torch.Tensor) -> torch.Tensor:
    """ops.member_sorted on tensors: bool[Q], hit[i] = q[i] is in sorted_wl.  sorted_wl must be ascending as uint32; it is
    checked as the host form checks it (one 8-byte wait), and an unsorted whitelist raises the same error."""
    _ready()
    _check(sorted_wl, "sorted_wl", BARCODE_DTYPES)
    _check(q, "q", BARCODE_DTYPES)
    Q, W = q.numel(), sorted_wl.numel()
    hit = torch.empty(Q, dtype=torch.bool, device=q.device)
    if Q:
        with torch.cuda.device(q.device):
            check(lib().bdg_dev_whitelist_check(_ptr(sorted_wl), W, _stream()))
            check(lib().bdg_dev_member_sorted(_ptr(sorted_wl), W, q.data_ptr(), Q, hit.data_ptr(), _stream()))
    return hit


def nearest_bounded(q: torch.Tensor, targets_in_order: torch.Tensor, max_d: int = 2):
    """ops.nearest_bounded on tensors: (argmin int32[Q], dist uint8[Q]), the first index of the minimum plain edit distance over
    the targets in their given order, kept when it is <= max_d; -1 / 255 otherwise."""
    _ready()
    _check(q, "q", BARCODE_DTYPES)
    _check(targets_in_order, "targets_in_order", BARCODE_DTYPES)
    Q, W, dev = q.numel(), targets_in_order.numel(), q.device
    am = torch.empty(Q, dtype=torch.int32, device=dev)
    dist = torch.empty(Q, dtype=torch.uint8, device=dev)
    if Q:
        keys = torch.empty(Q, dtype=torch.int32, device=dev)      # the packed (distance, index) minimum of every query
        with torch.cuda.device(dev):
            check(lib().bdg_dev_nearest_bounded(q.data_ptr(), Q, _ptr(targets_in_order), W, int(max_d), keys.data_ptr(), am.data_ptr(),
                                                dist.data_ptr(), _stream()))
    return am, dist


def _int32_sized(t, name):
    if t.numel() >= 1 << 31:
        raise ValueError("%s has %d entries; the hit indices are int32, so fewer than 2^31 are allowed" % (name, t.numel()))


def _kmer_query(call, q, n_known, min_kmers, cap, hint=None):
    """ops._kmer_query on tensors: the hits land in tensors sized for `cap` (returned as views of their first `hits` rows).  A
    first guess that is too small costs one repeated launch with the exact size; hint carries the room needed from call to call."""
    _check(q, "q", BARCODE_DTYPES)
    _int32_sized(q, "q")
    Q, dev = q.numel(), q.device
    if cap is None:
        cap = hint[0] if hint and hint[0] else max(1 << 16, min(4 * n_known, 2048 * max(Q, 1)))
    for attempt in range(2):
        hq = torch.empty(cap, dtype=torch.int32, device=dev)
        hw = torch.empty(cap, dtype=torch.int32, device=dev)
        cnt = torch.empty(cap, dtype=torch.uint8, device=dev)
        pos = torch.empty((cap, 11), dtype=torch.uint8, device=dev)
        total = C.c_size_t(0)
        with torch.cuda.device(dev):
            rc = call(_ptr(q), Q, int(min_kmers), cap, _ptr(hq), _ptr(hw), _ptr(cnt), _ptr(pos), C.byref(total), _stream())
        if rc == _lib.BDG_ERR_CAPACITY and attempt == 0:
            cap = int(total.value)
            continue
        check(rc)
        n = int(total.value)
        if hint is not None:
            hint[0] = max(1 << 16, n + n // 8)
        return hq[:n], hw[:n], cnt[:n], pos[:n]


def kmer_score(q: torch.Tensor, wl: torch.Tensor, min_kmers: int = 1, cap: int | None = None):
    """ops.kmer_score on tensors: (hit_q int32, hit_w int32, cnt uint8, pos uint8[hits, 11]) for every (query, string) pair with
    cnt >= min_kmers, order unspecified.  A one-off index: posting lists from 64 queries upwards, as bdg_kmer_score."""
    _ready()
    _check(wl, "wl", BARCODE_DTYPES)
    _int32_sized(wl, "wl")
    L, w = lib(), wl
    return _kmer_query(lambda *a: L.bdg_dev_kmer_score(a[0], a[1], _ptr(w), w.numel(), *a[2:]), q, wl.numel(), min_kmers, cap)


class KmerIndex(ops.KmerIndex):
    """ops.KmerIndex built from a tensor of known strings on the first device: query(q, min_kmers, cap) takes and returns tensors
    (see kmer_score); info() / free() as there.  The index stays on the device it was built on, which must still be the first
    device given to badger_b200.init when it is queried."""

    def __init__(self, known: torch.Tensor):
        _ready()
        _check(known, "known", BARCODE_DTYPES)
        _int32_sized(known, "known")
        self.size = int(known.numel())
        self._h = C.c_void_p()
        with torch.cuda.device(known.device):
            check(lib().bdg_dev_kmer_index_create(_ptr(known), self.size, _stream(), C.byref(self._h)))
        self._room = [0]

    def query(self, q: torch.Tensor, min_kmers: int = 1, cap: int | None = None):
        if self._h is None:
            raise ValueError("the index was freed")
        L = lib()
        return _kmer_query(lambda *a: L.bdg_dev_kmer_index_query(self._h, *a), q, self.size, min_kmers, cap, self._room)
