"""The correction step over a torch.distributed process group, one process per GPU: every rank keeps its own reads.

    every rank                                   what crosses between the ranks
      device.dedup_reads of its own reads          -
      its distinct list, counts, first sightings   all-gather (sizes, then the three lists padded to the longest)
      bdg_dev_dedup_merge                          -   (the global distinct set, the same on every rank; the rank's read map
                                                        now points at global first-seen positions)
      device.edges, part `rank` of `world`         all-reduce of the edge count; the edges stay on the rank that found them
      pipeline.select_centres                      -   (identical inputs on every rank: identical centres)
      cluster_levels: mark, two rounds             all-reduce of the levels (min), then per round of the claims (min / max)
      --high_sens on rank 0                        broadcast of the patched node -> centre array
      bdg_dev_assign_reads32 of its own rows       all-reduce of the rows with a centre

Nothing per read is exchanged.  Concatenated in rank order, the results equal those of device.assign_packed (and
pipeline.assign_packed(form="u32")) run in one process on the concatenation of the ranks' inputs in rank order.

`Tally` is the same step for reads that every rank adds in batches (device.Tally on each rank):

    every rank                                   what crosses between the ranks
      add: bdg_dev_tally_add of its own batches    -   (rank-local, any number of batches)
      finish: bdg_tally_info                       all-gather of the status, set size, rows, valid rows and scalar arguments
      bdg_dev_tally_copy of its running set        all-gather of the sets padded to the longest (20 B per entry per rank)
      bdg_dev_tally_merge_parts, bdg_dev_tally_finish   -   (the union in rank-major order, the same on every rank)
      run_stages: edges, centres, rounds, --high_sens   as for assign_packed above
      assign: bdg_dev_assign_lookup32 of any rows  -   (rank-local)

Every call of assign_packed, and Tally.finish, is collective: all ranks of the group make it, with the same scalar arguments.
Which collectives run depends only on those arguments and on values reduced over the group, never on a rank's own reads, so a rank
with no rows, or with no valid row, takes part like any other.  Collectives run on CUDA tensors in the order of torch.cuda.current_stream() (NCCL or gloo).
"""
from __future__ import annotations

import ctypes as C
import time

import numpy as np
import torch
import torch.distributed as dist

from . import _lib, pipeline
from . import device as bd
from ._lib import check, lib

ROUNDS = 2          # barcode_graph.py:279-301 runs two rounds


class _Group:
    """Rank, world size and the collectives of one call; without an initialised process group a world of one, whose collectives
    return their input.  `traffic` counts the bytes every collective delivered to this rank, by name."""

    def __init__(self, group, traffic=None):
        self.on = dist.is_available() and dist.is_initialized()
        self.pg = group
        self.rank = dist.get_rank(group) if self.on else 0
        self.world = dist.get_world_size(group) if self.on else 1
        self.traffic = traffic if traffic is not None else {}

    def _count(self, name, nbytes):
        self.traffic[name] = self.traffic.get(name, 0) + int(nbytes)

    def all_gather(self, t, name):
        """[world, *t.shape]: the tensors of all ranks in rank order."""
        out = torch.empty((self.world,) + tuple(t.shape), dtype=t.dtype, device=t.device)
        if self.on:
            dist.all_gather(list(out.unbind(0)), t, group=self.pg)
        else:
            out[0].copy_(t)
        self._count(name, out.numel() * out.element_size())
        return out

    def all_reduce(self, t, op, name):
        if self.on:
            dist.all_reduce(t, op=op, group=self.pg)
        self._count(name, t.numel() * t.element_size())
        return t

    def broadcast_from_first(self, t, name):
        if self.on:
            dist.broadcast(t, src=dist.get_global_rank(self.pg, 0) if self.pg is not None else 0, group=self.pg)
        self._count(name, t.numel() * t.element_size())
        return t


def _lists(rm, dev):
    """int32[3, n]: the rank's distinct barcodes ascending, their counts and their local first-seen positions."""
    n = rm.n_distinct
    out = torch.empty((3, n), dtype=torch.int32, device=dev)
    if n:
        sp = rm.sorted_pos                                            # first-seen -> ascending position
        out[0] = rm.sorted_distinct.view(torch.int32)
        out[1, sp] = rm.counts.to(torch.int32)
        out[2, sp] = torch.arange(n, dtype=torch.int32, device=dev)
    return out


def dedup_merge(rm, group=None, *, _g=None):
    """The distinct barcodes of every rank's read map `rm` (device.dedup_reads) merged into the global ones: a DeviceReadMap
    whose distinct / counts / sorted_pos / sorted_distinct are those of one dedup over the concatenation of all ranks' reads in
    rank order (the same on every rank), and whose read map holds this rank's rows.  rm's token dies.  Returns (merged, valid
    reads of all ranks, rows of all ranks); merged is None on every rank when no rank has a valid read."""
    g = _g or _Group(group)
    dev = bd._device()
    local = _lists(rm, dev)
    meta = torch.tensor([rm.n_distinct, rm.n_valid, rm.rows], dtype=torch.int64, device=dev)
    metas = g.all_gather(meta, "sizes").cpu()                         # host wait: the sizes decide the shapes below
    sizes = [int(x) for x in metas[:, 0]]
    total_valid, total_rows = int(metas[:, 1].sum()), int(metas[:, 2].sum())
    if total_valid == 0:
        return None, total_valid, total_rows
    width = max(sizes)
    mine = torch.zeros((3, width), dtype=torch.int32, device=dev)
    mine[:, :rm.n_distinct] = local
    parts = g.all_gather(mine, "lists")                               # [world, 3, width]
    base, row = parts.data_ptr(), 4 * width
    starts = (C.c_size_t * g.world)(*[3 * width * p for p in range(g.world)])
    n, tok = C.c_size_t(0), C.c_ulonglong(0)
    with torch.cuda.device(dev):
        check(lib().bdg_dev_dedup_merge(rm.token, base, base + row, base + 2 * row, starts, (C.c_size_t * g.world)(*sizes), g.world,
                                        g.rank, C.byref(n), C.byref(tok), bd._stream()))
    return bd.DeviceReadMap(int(n.value), rm.n_valid, rm.rows, int(tok.value), rm.dtype), total_valid, total_rows


def cluster_levels(sorted_distinct: torch.Tensor, ea: torch.Tensor, eb: torch.Tensor, centres, rounds: int = ROUNDS, *, group=None,
                   _g=None):
    """barcode_graph.py:279-301 over the union of the ranks' edge lists (every rank passes its own; each edge on one rank only),
    with the nodes (sorted_distinct, the same on every rank) and the centres (barcode values, the same on every rank) replicated.
    Returns (centre_idx int32[N], level uint8[N]) tensors, equal on every rank: as ops.cluster_levels, except that level 254 marks
    the nodes with an edge that no round reached.  The claims of every round are reduced over the group (minimum and maximum of
    the claiming centres), which is the reference's same-round conflict rule over the union."""
    g = _g or _Group(group)
    bd._check(sorted_distinct, "sorted_distinct", bd.BARCODE_DTYPES)
    bd._check(ea, "ea", (sorted_distinct.dtype,))
    bd._check(eb, "eb", (sorted_distinct.dtype,))
    dev, N, E = sorted_distinct.device, sorted_distinct.numel(), ea.numel()
    if eb.numel() != E:
        raise ValueError("ea has %d edges, eb %d" % (E, eb.numel()))
    cen = torch.from_numpy(np.ascontiguousarray(centres, dtype=np.uint32).view(np.int32)).to(dev)
    ci = torch.empty(N, dtype=torch.int32, device=dev)
    lv = torch.empty(N, dtype=torch.uint8, device=dev)
    cmin, cmax = torch.empty_like(ci), torch.empty_like(ci)
    ia, ib = torch.empty(E, dtype=torch.int32, device=dev), torch.empty(E, dtype=torch.int32, device=dev)
    bad = torch.zeros(1, dtype=torch.int32, device=dev)
    L, st, p = lib(), bd._stream(), bd._ptr
    with torch.cuda.device(dev):
        check(L.bdg_dev_cluster_init(sorted_distinct.data_ptr(), N, p(cen), cen.numel(), ci.data_ptr(), lv.data_ptr(), cmin.data_ptr(),
                                     cmax.data_ptr(), st))
        check(L.bdg_dev_index_edges(sorted_distinct.data_ptr(), N, p(ea), p(eb), E, p(ia), p(ib), st))
        check(L.bdg_dev_cluster_mark(p(ia), p(ib), E, lv.data_ptr(), bad.data_ptr(), st))
        g.all_reduce(lv, dist.ReduceOp.MIN, "levels")                 # 255 -> 254 wherever any rank has an edge; centres keep 0
        g.all_reduce(bad, dist.ReduceOp.MAX, "levels")
        for r in range(1, int(rounds) + 1):
            check(L.bdg_dev_cluster_claim(p(ia), p(ib), E, r, ci.data_ptr(), lv.data_ptr(), cmin.data_ptr(), cmax.data_ptr(), st))
            g.all_reduce(cmin, dist.ReduceOp.MIN, "claims")
            g.all_reduce(cmax, dist.ReduceOp.MAX, "claims")
            check(L.bdg_dev_cluster_resolve(ci.data_ptr(), lv.data_ptr(), cmin.data_ptr(), cmax.data_ptr(), N, r, st))
    if int(bad.item()):
        raise _lib.BadgerB200Error(_lib.BDG_ERR_ARG, "an edge end point is not in the barcode array")
    return ci, lv


class _GroupStages:
    """The stages of pipeline.run_stages over the group: part `rank` of `world` of the edges on every rank and an all-reduce of
    their count, the clustering rounds of cluster_levels, --high_sens on rank 0 and a broadcast.  `g` holds the group of one
    call; with timings, every stage ends in a device synchronise."""

    def __init__(self, group, timings):
        self.g = _Group(group, timings.setdefault("collective_bytes", {}) if timings is not None else None)
        self.sync = (lambda: torch.cuda.synchronize(bd._device())) if timings is not None else None

    def edges(self, rm, threshold):
        g = self.g
        self.a, self.b, _ = bd.edges(rm.sorted_distinct, threshold, part=g.rank, nparts=g.world)
        n_edges = g.all_reduce(torch.tensor([self.a.numel()], dtype=torch.int64, device=bd._device()), dist.ReduceOp.SUM, "counts")
        return int(n_edges.item())

    def rounds(self, rm, centres, want_ci):
        ci, lv = cluster_levels(rm.sorted_distinct, self.a, self.b, centres, _g=self.g)
        del self.a, self.b
        return ci, int(((lv != 255) & (lv != 0)).sum().item())

    def patch(self, ci, rm, centre_order):
        if self.g.rank == 0:
            ci.copy_(torch.from_numpy(pipeline.high_sens_patch(ci.cpu().numpy(), rm.host.sorted_distinct, rm.host.sorted_pos, centre_order)))
        return self.g.broadcast_from_first(ci, "high_sens")


def assign_packed(ranks: torch.Tensor, valid: torch.Tensor | None = None, *, threshold, n_cells, interval=25, whitelist_sorted=None,
                  true_barcodes=None, high_sens=False, centre_order=None, group=None, timings=None):
    """device.assign_packed over the ranks of `group` (None: the default group; no initialised process group: a world of one).
    Called on every rank with that rank's reads (ranks / valid: CUDA tensors on the first device given to badger_b200.init, as
    for device.assign_packed) and the same scalar arguments; whitelist_sorted and true_barcodes are the same on every rank.
    Returns ((centre, has_centre), info) for the rank's own rows.  Concatenated in rank order, the results of all ranks equal
    device.assign_packed run in one process on the concatenation of their inputs in rank order (first-seen order therefore
    starts with rank 0's reads), and `info` - the same on every rank - equals its `info`.

    With high_sens, rank 0 runs the per-barcode --high_sens work of pipeline.assign_packed on the host and broadcasts the result;
    centre_order="set" is the set order of rank 0's process.  timings: a dict that receives the host time of every stage, each
    stage ended by a device synchronise, and under "collective_bytes" the bytes each kind of collective delivered to this rank."""
    bd._ready()
    bd._check(ranks, "ranks", bd.BARCODE_DTYPES)
    bd._check_whitelist(whitelist_sorted)
    true_barcodes = bd._true_barcodes(true_barcodes)
    T = timings if timings is not None else {}
    stages = _GroupStages(group, timings)
    g, R, dev = stages.g, ranks.numel(), ranks.device

    t0 = time.perf_counter()
    rm = bd.dedup_reads(ranks, valid)
    pipeline._tick(T, "dedup_first_seen", t0, stages.sync)

    t0 = time.perf_counter()
    merged, total_valid, total_rows = dedup_merge(rm, _g=g)
    pipeline._tick(T, "exchange_merge", t0, stages.sync)
    info = {"reads": total_rows, "valid_reads": total_valid}
    if merged is None:
        return bd._zeros(ranks), info

    def gather(ci):
        centre, has = bd._zeros(ranks)
        if rm.n_valid:
            with torch.cuda.device(dev):
                check(lib().bdg_dev_assign_reads32(merged.token, ci.data_ptr(), merged.n_distinct, centre.data_ptr(), has.data_ptr(), R, None,
                                                   bd._stream()))
        n_assigned = g.all_reduce(has.sum(dtype=torch.int64).reshape(1), dist.ReduceOp.SUM, "counts")
        return (centre, has), int(n_assigned.item())

    out = pipeline.run_stages(merged, info, T, stages, gather, threshold=threshold, n_cells=n_cells, interval=interval,
                              whitelist_sorted=whitelist_sorted, true_barcodes=true_barcodes, high_sens=high_sens,
                              centre_order=centre_order, centres_above=bd.centres_above)
    return out, info


class Tally(bd.Tally):
    """device.Tally over the ranks of `group` (None: the default group; no initialised process group: a world of one, which
    equals device.Tally).  Every rank adds its own batches; finish merges the ranks' running sets on the device.

    add(ranks, valid=None) and assign(ranks, valid=None) are rank-local, as in device.Tally: a rank may add any number of batches
    (none too), and assign any rows, another rank's included.  finish(...) is collective: every rank of the group calls it with the
    same scalar arguments, the same whitelist and the same true barcodes.  The result equals pipeline.assign_packed(form="u32")
    run in one process on the rank-major concatenation of the batches: rank 0's batches in add order, then rank 1's, ...  So
    first-seen order, count ties and the n_cells cutoff start with rank 0's first batch; with high_sens, rank 0 patches and
    broadcasts, and centre_order="set" is the set order of rank 0's process.  `info` is that process's info on every rank, except
    "assigned_reads": 0 after finish, then the rows with a centre of this rank's assign calls (summed over the ranks: the
    one-process figure).  finish's timings: as for assign_packed, with "exchange_merge", "tally_finish", "edges", "centres",
    "cluster", "high_sens", "gather" and "collective_bytes".

    A refusal is decided from data that is the same on every rank: a rank-local problem (a freed tally, a bad argument, a finish
    on some ranks only) travels in the first all-gather of finish, and every rank raises."""

    def __init__(self, group=None):
        super().__init__()
        self._group = group
        self._totals = None           # (rows, valid rows) of all ranks once finish merged the sets

    def _stages(self, timings):
        return _GroupStages(self._group, timings)

    def _read_map(self, n_distinct, n_valid, token):
        return bd.DeviceReadMap(n_distinct, n_valid, 0, token, torch.int32)

    def _close(self, stages, T, args):
        """Steps: (1) all-gather of every rank's status, set size, rows and scalar arguments; (2) all-gather of the sets
        (bdg_dev_tally_copy, padded to the longest); (3) bdg_dev_tally_merge_parts; (4) bdg_dev_tally_finish.  Returns the rows
        and valid rows of all ranks."""
        g, dev, L = stages.g, bd._device(), lib()

        t0 = time.perf_counter()
        err, status, own = None, 0, [0, 0, 0]
        scalars = [0, 0, 0, 0]
        try:
            h = self._handle()
            scalars = [int(args["threshold"]), int(args["n_cells"]), int(args["interval"]), int(bool(args["high_sens"]))]
            bd._check_whitelist(args["whitelist_sorted"])
            args["true_barcodes"] = bd._true_barcodes(args["true_barcodes"])
            n, rows, valid = C.c_size_t(0), C.c_ulonglong(0), C.c_ulonglong(0)
            check(L.bdg_tally_info(h, C.byref(n), C.byref(rows), C.byref(valid)))
            own = [int(n.value), int(rows.value), int(valid.value)] if self._totals is None else [0, *self._totals]
        except _lib.BadgerB200Error as e:
            err, status = e, 2
        except (TypeError, ValueError) as e:
            err, status = e, 1
        meta = torch.tensor([status, int(self._totals is not None)] + own + scalars, dtype=torch.int64, device=dev)
        metas = g.all_gather(meta, "sizes").cpu()                     # host wait: the sizes decide the shapes below
        refused = [r for r in range(g.world) if metas[r, 0]]
        if refused:
            if err is not None:
                raise err
            msg = "finish was refused on rank(s) %s" % refused
            if int(metas[refused[0], 0]) == 2:
                raise _lib.BadgerB200Error(_lib.BDG_ERR_ARG, msg)
            raise ValueError(msg)
        if not bool((metas[:, 5:] == metas[0, 5:]).all()):
            raise ValueError("the ranks called finish with different threshold / n_cells / interval / high_sens")
        if not bool((metas[:, 1] == metas[0, 1]).all()):
            raise ValueError("finish ran before on some ranks only")
        if self._totals is not None:                                  # a second finish: the handle holds the union already
            total_rows, total_valid = int(metas[0, 3]), int(metas[0, 4])
        else:
            sizes = [int(x) for x in metas[:, 2]]
            rows = [int(x) for x in metas[:, 3]]
            total_rows, total_valid = sum(rows), int(metas[:, 4].sum())
            if total_valid:
                width = max(sizes)
                key = torch.empty(width, dtype=torch.int32, device=dev)
                cnt = torch.empty(width, dtype=torch.int64, device=dev)
                first = torch.empty(width, dtype=torch.int64, device=dev)
                with torch.cuda.device(dev):
                    check(L.bdg_dev_tally_copy(h, key.data_ptr(), cnt.data_ptr(), first.data_ptr(), bd._stream()))
                keys, cnts, firsts = (g.all_gather(x, "sets") for x in (key, cnt, first))     # [world, width] each
                offsets = np.concatenate([[0], np.cumsum(rows)[:-1]]).tolist()
                with torch.cuda.device(dev):
                    check(L.bdg_dev_tally_merge_parts(h, keys.data_ptr(), cnts.data_ptr(), firsts.data_ptr(),
                                                      (C.c_size_t * g.world)(*[width * p for p in range(g.world)]),
                                                      (C.c_size_t * g.world)(*sizes), (C.c_ulonglong * g.world)(*offsets), g.world,
                                                      g.rank, total_rows, total_valid, bd._stream()))
            self._totals = (total_rows, total_valid)
        pipeline._tick(T, "exchange_merge", t0, stages.sync)

        _, _, n_distinct, token = super()._close(stages, T, args)    # a merged count of 2^32 or more: refused on every rank
        return total_rows, total_valid, n_distinct, token
