"""Array form of the correction step (reference badger.py:120-129 with barcode_graph.py:192-410 behind it): packed
barcodes per read in, cluster-centre barcode per read out, every stage on the GPU operators, no per-read Python.

    read barcodes (uint32 per row + valid mask)
      -> ops.dedup_reads                 barcode_graph.py:192-204   valid rows compacted on the device; distinct barcodes in
                                                                    first-seen order, counts; the read map STAYS on the device
      -> ops.edges_handle                index.py:77-93 + barcode_graph.py:224-249   every claimed GPU builds its part; edges stay there
      -> ops.centres_above + walk_centres   barcode_graph.py:252-277   cutoff, count-ordered head of the list and its whitelist hits on the GPU
      -> EdgeHandle.cluster_resident     barcode_graph.py:279-301   two rounds, same-round conflicts evict (parts gathered over NVLink)
      -> ops.nearest_bounded             barcode_graph.py:370-385   only with high_sens; patches the node -> centre array
      -> ops.assign_reads32              barcode_graph.py:322-329,395-404   centre of every row: gather kernel over the resident read map

The string-based mirror (``BarcodeGraph`` + ``badger.py``) gives the same assignments; this module exists for callers
that already hold packed barcodes and for the reads/s figure of ``bench.py``.  ``Tally`` is the same step for reads that
arrive in batches: the dedup runs batch by batch into a running distinct set on the device, and the per-read gather looks
every row's barcode up among the nodes.
"""
from __future__ import annotations

import ctypes as C
import time

import numpy as np

from . import _lib, ops
from ._lib import check, lib, ptr
from .barcode_graph import _unrank_many
from .common import rank

NONE = ops.NONE                           # "no centre" marker in the uint64 result (every uint32 is a valid barcode)


class _Token:
    """Stands in for the whitelist set the string API passes around (truthy, compared by identity)."""

    def __bool__(self):
        return True


def select_centres(rm, n_cells, interval, whitelist_sorted, true_barcodes, centres_above=ops.centres_above):
    """barcode_graph.py:252-277 with the counting, the count-ordered head of the barcode list and its whitelist membership on
    the device (centres_above, and ops.centres_rest if the top-up loop has to go below the cutoff): no per-barcode array is
    downloaded."""
    from statistics import StatisticsError
    from .barcode_graph import walk_centres
    if rm.n_distinct == 0 or n_cells <= 0:
        raise StatisticsError("mean requires at least one data point")
    tb = None if true_barcodes is None else [int(x) for x in true_barcodes]
    cutoff, top, _, hits = centres_above(rm, n_cells, None if tb else whitelist_sorted)
    have_list = whitelist_sorted is not None
    if hits is None and have_list and not tb:
        hits = np.zeros(0, bool)
    return walk_centres(rm.n_distinct, n_cells, interval, top, hits, tb, have_list,
                        lambda need: ops.centres_rest(rm, cutoff, int(need) + 1))


def assign_packed(ranks, valid=None, *, threshold, n_cells, interval=25, whitelist_sorted=None, true_barcodes=None,
                  high_sens=False, centre_order=None, timings=None, form="u64"):
    """Returns (centre uint64[R], info) - centre[i] == pipeline.NONE where the reference would write ``*`` - or, with
    form="u32", ((centre uint32[R], has_centre uint8[R]), info): 5 instead of 8 bytes per row cross PCIe.

    ranks / valid: packed barcode and validity per read (valid=None: all valid); whitelist_sorted: ascending uint32 array
    or None; true_barcodes: iterable of packed centres or None (badger.py --true_barcodes); centre_order: order in which
    --high_sens tries the centres (the reference iterates a Python set, barcode_graph.py:372; default: ascending; "set":
    the iteration order of that very set of strings in this process, which is what badger_b200.BarcodeGraph meets too).

    Without high_sens nothing per-barcode ever reaches the host: the distinct barcodes, their counts, the edges, the
    clustering result and the read map stay on the device between the stages.  (badger_b200.device.assign_packed is the
    same step with the per-read arrays in CUDA tensors.)"""
    T = timings if timings is not None else {}

    def result(c32, has):
        return (c32, has) if form == "u32" else ops.widen(c32, has)

    ranks = np.ascontiguousarray(ranks, dtype=np.uint32)
    R = ranks.size
    info = {"reads": int(R)}
    if R == 0:
        info["valid_reads"] = 0
        return result(*_zeros(ranks)), info

    t0 = time.perf_counter()
    rm = ops.dedup_reads(ranks, valid)                    # valid rows compacted on the device; everything stays there
    _tick(T, "dedup_first_seen", t0)
    info["valid_reads"] = int(rm.n_valid)
    if rm.n_valid == 0:
        return result(*_zeros(ranks)), info

    def gather(ci):
        c32, has, n_assigned = ops.assign_reads32(rm, ci)     # per-read gather on the device
        return result(c32, has), n_assigned

    return run_stages(rm, info, T, _OneProcess(), gather, threshold=threshold, n_cells=n_cells, interval=interval,
                      whitelist_sorted=whitelist_sorted, true_barcodes=true_barcodes, high_sens=high_sens, centre_order=centre_order,
                      centres_above=ops.centres_above), info


def _tick(T, name, t0, sync=None):
    """Adds the host time since t0 to T[name]; sync, when given, waits for the device first."""
    if sync is not None:
        sync()
    T[name] = T.get(name, 0.0) + time.perf_counter() - t0


def _zeros(ranks):
    """The result of rows none of which has a centre: (centre uint32[R], has_centre uint8[R]), all zero."""
    return np.zeros(ranks.size, np.uint32), np.zeros(ranks.size, np.uint8)


class Tally:
    """The correction step over reads that arrive in batches (include/badger_b200.h bdg_tally_*): `add` batches 0 ... B-1 in order,
    `finish` once, then `assign` any rows.  The result of `assign` equals, element for element, what assign_packed(form="u32")
    gives those rows when it runs on the concatenation of the added batches, and `finish` returns its `info` (with
    "assigned_reads" summed over the assign calls).  Only the distinct barcodes, their counts and first sightings are kept
    between batches, on the device; the device memory per read grows with the batch, not with the total, and the total may
    exceed the 2^31 reads of one assign_packed call (each batch stays below 2^31 rows).

    Every add and finish is a dedup call: it kills the read map of an outstanding ops.dedup_reads token, and a later dedup call
    (another tally's add, assign_packed, ...) makes `assign` raise until `finish` runs again."""

    _centres_above = staticmethod(ops.centres_above)
    _zeros = staticmethod(_zeros)

    def __init__(self):
        self._h = C.c_void_p()
        check(lib().bdg_tally_create(C.byref(self._h)))
        self.rows = 0
        self.info = None              # finish's result: `info` of the one-call step
        self._rm = None               # the read map finish installed (None: no valid read was added)
        self._ci = None               # with high_sens, the patched node -> centre array; None: the clustering left on the device

    def _handle(self):
        if self._h is None or not self._h.value:
            raise ValueError("the tally was freed")
        return self._h

    @staticmethod
    def _rows(ranks, valid):
        r = np.ascontiguousarray(ranks, dtype=np.uint32)
        return r, ops._mask(valid, r.size)

    def add(self, ranks, valid=None) -> int:
        """Count one batch (packed barcodes per row; valid: mask or None for all rows).  Returns its number of valid rows."""
        r, v = self._rows(ranks, valid)
        nv = C.c_size_t(0)
        check(lib().bdg_tally_add(self._handle(), ptr(r), ptr(v) if v is not None else None, r.size, C.byref(nv)))
        self.rows += r.size
        return int(nv.value)

    def finish(self, *, threshold, n_cells, interval=25, whitelist_sorted=None, true_barcodes=None, high_sens=False, centre_order=None,
               timings=None) -> dict:
        """The stages after the dedup (run_stages, arguments as for assign_packed) over the counted batches.  The clustering
        result stays for `assign`.  Returns `info`; no batch can be added afterwards."""
        T = timings if timings is not None else {}
        args = dict(threshold=threshold, n_cells=n_cells, interval=interval, whitelist_sorted=whitelist_sorted,
                    true_barcodes=true_barcodes, high_sens=high_sens, centre_order=centre_order)
        stages = self._stages(timings)
        rows, n_valid, n_distinct, token = self._close(stages, T, args)
        self.info = info = {"reads": int(rows), "valid_reads": int(n_valid)}
        self._rm, self._ci = None, None
        if n_valid == 0:
            return info
        rm = self._read_map(n_distinct, n_valid, token)

        def keep(ci):
            self._ci = None if ci is None else self._upload(ci)
            return None, 0

        run_stages(rm, info, T, stages, keep, centres_above=self._centres_above, **args)
        self._rm = rm
        return info

    def _stages(self, timings):
        return _OneProcess()

    def _close(self, stages, T, args):
        """Ends the counting: (rows, valid rows, distinct barcodes, token of the read map) of the counted batches.  args: the
        arguments of finish, which a form may check and normalise in place."""
        t0 = time.perf_counter()
        n, nv, tok = C.c_size_t(0), C.c_size_t(0), C.c_ulonglong(0)
        self._finish_call(n, nv, tok)
        _tick(T, "tally_finish", t0, stages.sync)
        return self.rows, int(nv.value), int(n.value), int(tok.value)

    def _finish_call(self, n, nv, tok):
        check(lib().bdg_tally_finish(self._handle(), C.byref(n), C.byref(nv), C.byref(tok)))

    def _read_map(self, n_distinct, n_valid, token):
        return ops.ReadMap(n_distinct, n_valid, 0, token)

    def _upload(self, ci):
        return np.ascontiguousarray(ci, dtype=np.int32)

    def assign(self, ranks, valid=None):
        """(centre uint32[R], has_centre uint8[R]) for the rows of `ranks`, any batching.  ValueError when a valid row's barcode
        was never added.  With high_sens the patched node -> centre array is copied to the device with every call (the tensor
        form, device.Tally, uploads it once)."""
        if self.info is None:
            raise ValueError("assign before finish")
        r, v = self._rows(ranks, valid)
        if self._rm is None:                                  # nothing was counted: only rows without a barcode can be assigned
            n_valid = len(r) if v is None else int((v != 0).sum())
            if n_valid:
                raise ValueError("%d valid rows have a barcode that was never added" % n_valid)
            return self._zeros(r)
        centre, has, n_assigned, n_missing = self._lookup(self._rm, r, v)
        if n_missing:
            raise ValueError("%d valid rows have a barcode that was never added" % n_missing)
        self.info["assigned_reads"] += n_assigned
        return centre, has

    def _lookup(self, rm, r, v):
        """(centre, has_centre, rows with a centre, valid rows whose barcode is not a node)."""
        out = ops._pinned.array(r.size, np.uint32, eager=False)
        has = ops._pinned.array(r.size, np.uint8, eager=False)
        na, nm = C.c_size_t(0), C.c_size_t(0)
        ci = self._ci
        check(lib().bdg_assign_lookup32(rm.token, ptr(ci) if ci is not None else None, rm.n_distinct, ptr(r), ptr(v) if v is not None else None,
                                        r.size, ptr(out), ptr(has), C.byref(na), C.byref(nm)))
        return out, has, int(na.value), int(nm.value)

    def free(self):
        if self._h is not None and self._h.value and _lib._lib is not None:
            lib().bdg_tally_free(self._h)
        self._h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def run_stages(rm, info, T, stages, gather, *, threshold, n_cells, interval, whitelist_sorted, true_barcodes, high_sens, centre_order,
               centres_above):
    """The stages after the dedup (or the merge of the ranks' barcodes) of a read map `rm` with at least one valid read: edges,
    centres, clustering, --high_sens, and last `gather(centre_idx)` -> (result, rows with a centre) over the read map, with
    centre_idx None for the clustering left on the device.  `stages` builds the edges and runs the rounds and the patch:
    _OneProcess, or distributed._GroupStages over a process group; its `sync` (None: none) ends every timed stage.  Fills `info`
    and the timings `T`; returns what `gather` returned first.  centres_above is ops.centres_above or a function of the same
    signature that takes the whitelist in another form."""
    def tick(name, t0):
        _tick(T, name, t0, stages.sync)

    t0 = time.perf_counter()
    n_edges = stages.edges(rm, threshold)
    info.update(distinct=int(rm.n_distinct), edges=int(n_edges))
    tick("edges", t0)

    t0 = time.perf_counter()
    centres = np.asarray(list(dict.fromkeys(select_centres(rm, n_cells, interval, whitelist_sorted, true_barcodes, centres_above))),
                         dtype=np.uint32)
    info["centres"] = int(centres.size)
    tick("centres", t0)

    t0 = time.perf_counter()
    ci, n_has_edge = stages.rounds(rm, centres, high_sens)
    # badger.py:131 `len(counts) - len(edges.keys())`: the keys are the nodes with an edge plus every centre cluster() touched
    info["disconnected"] = int(rm.n_distinct) - (int(n_has_edge) + int(centres.size))
    tick("cluster", t0)

    if high_sens:
        t0 = time.perf_counter()
        ci = stages.patch(ci, rm, centre_order)
        tick("high_sens", t0)

    t0 = time.perf_counter()
    out, n_assigned = gather(ci)
    info["assigned_reads"] = int(n_assigned)
    tick("gather", t0)
    return out


class _OneProcess:
    """The stages of run_stages in one process: the edges built on every claimed GPU from the distinct barcodes the read map
    keeps on the first one, the rounds over them (the node -> centre array stays on the device unless --high_sens patches it
    on the host).  The timings do not wait for the device."""

    sync = None

    def edges(self, rm, threshold):
        self.handle = ops.edges_handle_resident(rm, threshold)    # the ascending array is already on the device: no upload, peer copies to the other GPUs
        return self.handle.count

    def rounds(self, rm, centres, want_ci):
        if want_ci:
            ci, _, has_edge = self.handle.cluster_levels(centres, 2, want_has_edge=True)
            n_has_edge = int(has_edge.sum())
        else:
            ci, n_has_edge = None, self.handle.cluster_resident(centres, 2)
        self.handle.free()
        return ci, n_has_edge

    def patch(self, ci, rm, centre_order):
        return high_sens_patch(ci, rm.sorted_distinct, rm.sorted_pos, centre_order)


def high_sens_patch(ci, s, spos, centre_order):
    """barcode_graph.py:370-385 on node positions: every node without a centre (ci < 0) takes the nearest used centre within
    distance 2, tried in the order centre_order names (see assign_packed).  ci: the clustering result (int32[N], patched in
    place and returned); s: the distinct barcodes ascending; spos: their first-seen -> ascending positions."""
    todo = np.nonzero(ci < 0)[0]
    used_nodes = ops.sorted_unique(ci[ci >= 0])                              # set(assignments.values()), as nodes (ascending = by value)
    if centre_order is None:
        targets = s[used_nodes]
    elif isinstance(centre_order, str) and centre_order == "set":
        # the order the string route meets in this process: `set(assignments.values())` with the dict filled in
        # first-seen order of the distinct barcodes (barcode_graph.py:322-329,372).  Re-adding a member leaves a set's
        # table untouched, so the set of the first occurrences, added in that order, iterates identically.
        cfs = ci[spos]                                                       # centre node per distinct barcode, first-seen order
        vals = cfs[cfs >= 0]
        order = np.argsort(vals, kind="stable")                              # first occurrence of every value, in order of appearance
        sv = vals[order]
        head = np.ones(sv.size, bool)
        head[1:] = sv[1:] != sv[:-1]
        strs = _unrank_many(s[vals[np.sort(order[head])]])
        targets = np.asarray([rank(c, 16) for c in set(strs)], np.uint32)
    else:
        used = set(s[used_nodes].tolist())
        targets = np.asarray([c for c in centre_order if c in used], np.uint32)
    if todo.size and targets.size:
        am, _ = ops.nearest_bounded(s[todo], targets, 2)
        hit = am >= 0
        ci[todo[hit]] = np.searchsorted(s, targets[am[hit]]).astype(np.int32)
    return ci
