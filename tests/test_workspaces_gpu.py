"""The host-side state that ties the correction step's stages together: a clustering left on the device serves only the read map
its edges were built from, and bdg_shutdown returns every workspace, the merge's included."""
import ctypes as C
import gc

import numpy as np
import pytest
import torch

import badger_b200
from badger_b200 import _lib, ops, pipeline, synth
from badger_b200 import device as bd
from badger_b200 import distributed as bdist
from gpu_helpers import claimed

pytestmark = pytest.mark.gpu


def reads(seed, n_reads=200000, n_cells=300):
    rng = synth.rng_for(seed)
    wl = synth.make_whitelist(20000, rng)
    cells = synth.pick_cells(wl, n_cells, rng)
    obs, valid = synth.simulate_reads(cells, n_reads, 0.08, rng)
    return obs, valid, cells


def refused(rm):
    with pytest.raises(_lib.BadgerB200Error) as e:
        ops.assign_reads32(rm, None)
    assert e.value.code == _lib.BDG_ERR_ARG


def test_clustering_of_a_host_array_handle_does_not_serve_a_read_map(claimed):
    """A handle built from a host array with as many barcodes as the read map has: its clustering is not the read map's."""
    obs, valid, cells = reads(11)
    rm = ops.dedup_reads(obs, valid)
    s2 = np.arange(rm.n_distinct, dtype=np.uint32) * 3 + 1            # strictly increasing, not the read map's barcodes
    assert not np.array_equal(s2, rm.sorted_distinct)
    h = ops.edges_handle(s2, 1)
    h.cluster_resident(s2[:50], 2)
    h.free()
    refused(rm)
    # the read map itself is intact: its own graph clusters and gathers
    h = ops.edges_handle_resident(rm, 1)
    h.cluster_resident(cells, 2)
    h.free()
    c32, has, n = ops.assign_reads32(rm, None)
    assert c32.size == obs.size and 0 < n <= int(valid.sum())


def test_clustering_of_an_earlier_read_map_does_not_serve_a_later_one(claimed):
    """A handle built from read map 1, clustered after a second dedup call of the same size installed read map 2; and a tally,
    whose finish installs a read map and clusters its graph before assign."""
    obs, valid, cells = reads(12)
    rm1 = ops.dedup_reads(obs, valid)
    h = ops.edges_handle_resident(rm1, 1)
    s1 = rm1.sorted_distinct
    obs2 = obs ^ np.uint32(0x5)                                         # other barcodes, the same number of distinct ones
    rm2 = ops.dedup_reads(obs2, valid)
    assert rm2.n_distinct == rm1.n_distinct and not np.array_equal(rm2.sorted_distinct, s1)
    h.cluster_resident(cells, 2)
    h.free()
    refused(rm2)
    # a tally installs its own read map at finish and clusters that graph: assign serves it as before
    kw = dict(threshold=1, n_cells=300)
    (want_c, want_h), winfo = pipeline.assign_packed(obs, valid, form="u32", **kw)
    tally = pipeline.Tally()
    try:
        tally.add(obs, valid)
        tally.finish(**kw)
        c32, has = tally.assign(obs, valid)
    finally:
        tally.free()
    assert np.array_equal(c32, want_c) and np.array_equal(has, want_h) and tally.info == winfo


def dedup_and_merge(n):
    """bdg_dev_dedup_merge in a world of one over n distinct barcodes (an odd multiplier makes arange(n) n distinct values)."""
    L, dev = badger_b200.lib(), bd._device()
    x = (torch.arange(n, dtype=torch.int64, device=dev) * 2654435761) & 0xFFFFFFFF
    obs = torch.where(x >= 1 << 31, x - (1 << 32), x).to(torch.int32)
    del x
    rm = bd.dedup_reads(obs)
    assert rm.n_distinct == n
    lists = bdist._lists(rm, dev)
    base = lists.data_ptr()
    nd, mt = C.c_size_t(0), C.c_ulonglong(0)
    _lib.check(L.bdg_dev_dedup_merge(rm.token, base, base + 4 * n, base + 8 * n, (C.c_size_t * 1)(0), (C.c_size_t * 1)(n), 1, 0,
                                     C.byref(nd), C.byref(mt), bd._stream()))
    assert nd.value == n and mt.value != 0
    torch.cuda.synchronize(dev)


def test_shutdown_frees_the_merge_workspaces(claimed):
    """A merge over 5e7 distinct barcodes, then bdg_shutdown: the device memory the library held for the dedup and the merge is
    returned.  The reference reading is taken with no workspace held (right after a shutdown), once a small merge has loaded
    every module the large one runs.  The tolerance is below the smallest workspace of that size (5e7 x 4 B)."""
    L, dev = badger_b200.lib(), bd._device()

    def free_after_shutdown():
        gc.collect()
        torch.cuda.synchronize(dev)
        torch.cuda.empty_cache()
        L.bdg_shutdown()
        return torch.cuda.mem_get_info(dev)[0]

    dedup_and_merge(1000)
    free0 = free_after_shutdown()
    badger_b200.init()
    dedup_and_merge(50_000_000)
    free1 = free_after_shutdown()
    print("free device memory: %.3f GB before the dedup and merge, %.3f GB after bdg_shutdown" % (free0 / 1e9, free1 / 1e9))
    assert free0 - free1 < 128 << 20
