"""badger_b200.distributed.Tally, the batched correction step over a process group, against the one-process step on the rank-major
concatenation of every rank's batches (rank 0's batches in add order, then rank 1's, ...): the per-read results of every rank's
assign calls and `info` must equal pipeline.assign_packed(form="u32") there, element for element.

Worlds of 2 and 3 ranks run on gloo with every rank on the first GPU; a world of min(4, GPUs) ranks runs on NCCL with one GPU
per rank.  Each world is one set of spawned processes that runs every check and reports to the test; the reference runs on
rank 0 in the same process as that rank's tally, so that centre_order="set" meets the same set order."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import badger_b200
from badger_b200 import device as bd
from badger_b200 import distributed as bdist
from badger_b200 import ops, pipeline, synth
from badger_b200._lib import BDG_ERR_ARG, BDG_OK, BadgerB200Error
from gpu_helpers import ROOT, assert_world, claimed_without_group, cuda, dataset, host, run_world

TESTS = os.path.dirname(os.path.abspath(__file__))
pytestmark = pytest.mark.gpu

N_READS = 100000
N_CELLS = 300
CASES = [  # threshold, whitelist, valid mask, true barcodes, high_sens, centre_order, barcode dtype, how the reads are split
    (1, True, True, False, False, None, torch.int32, "uneven"),
    (2, False, False, False, False, None, torch.uint32, "first_empty"),
    (2, True, True, False, True, None, torch.int32, "uneven"),
    (2, False, True, True, True, "set", torch.int32, "last_invalid"),
    (3, True, True, False, False, None, torch.uint32, "uneven"),
    (3, False, True, True, False, None, torch.int32, "late_new"),
]


def bounds(split, world, n):
    """[lo, hi) of every rank: uneven weights 3, 1, 2, 3, 1, 2, ...; "first_empty" gives rank 0 no rows."""
    w = np.array([0 if (split == "first_empty" and r == 0) else (3, 1, 2)[r % 3] for r in range(world)], float)
    if world == 1:
        w[:] = 1
    cut = np.concatenate([[0], np.round(np.cumsum(w) / w.sum() * n)]).astype(int)
    return [(int(cut[r]), int(cut[r + 1])) for r in range(world)]


def batches(lo, hi, k, seed):
    """[lo, hi) cut into k uneven batches (k = 0: none)."""
    if k == 0 or hi == lo:
        return []
    rng = np.random.default_rng(seed)
    cut = np.sort(rng.integers(lo, hi + 1, k - 1))
    edges = np.concatenate([[lo], cut, [hi]]).astype(int)
    return [(int(a), int(b)) for a, b in zip(edges[:-1], edges[1:])]


def without_assigned(info):
    return {k: v for k, v in info.items() if k != "assigned_reads"}


# ---------------------------------------------------------------------------------------------------------------- the checks
def check_cases(rank, world, gather, record):
    for k, (t, use_wl, use_valid, use_tb, high_sens, order, dtype, split) in enumerate(CASES):
        wl, cells, obs, valid = dataset(700 + k, N_READS, N_CELLS)
        if split == "late_new":                               # barcodes first seen in the last rank's last batch
            fresh = synth.rng_for(5).integers(0, 1 << 32, 40, dtype=np.uint64).astype(np.uint32)
            obs = np.concatenate([obs, np.repeat(fresh, 3)])
            valid = np.concatenate([valid, np.ones(fresh.size * 3, bool)])
        b = bounds("first_empty" if split == "first_empty" else "uneven", world, obs.size)
        v = valid.copy()
        lo, hi = b[rank]
        if split == "last_invalid":                           # the last rank adds one batch, with no valid row
            v[b[-1][0]:] = False
            add_cuts = [(lo, hi)] if rank == world - 1 else batches(lo, hi, 2 + rank, k)
        else:
            add_cuts = batches(lo, hi, (1 + rank) % 4 + 1, 10 * k + rank)     # ranks add different numbers of batches
        wls = np.sort(wl)
        kw = dict(threshold=t, n_cells=N_CELLS, high_sens=high_sens, centre_order=order)
        tl = bdist.Tally()
        for a, z in add_cuts:
            tl.add(cuda(obs[a:z], dtype), cuda(v[a:z], torch.bool) if use_valid else None)
        info = tl.finish(whitelist_sorted=cuda(wls, dtype) if use_wl else None, true_barcodes=cuda(cells[:200], dtype) if use_tb else None,
                         **kw)
        c_parts, h_parts = [], []
        for a, z in batches(lo, hi, 3, 99 + k):               # an assign batching that differs from the add batching
            c, h = tl.assign(cuda(obs[a:z], dtype), cuda(v[a:z], torch.bool) if use_valid else None)
            ok_dtype = c.dtype == dtype and h.dtype == torch.bool and c.numel() == z - a
            c_parts.append(host(c)); h_parts.append(host(h))
        mine = dict(info)
        o_lo, o_hi = b[(rank + 1) % world]                    # another rank's rows
        oc, oh = tl.assign(cuda(obs[o_lo:o_hi], dtype), cuda(v[o_lo:o_hi], torch.bool) if use_valid else None)
        tl.free()
        cat = (lambda xs, dt: np.concatenate(xs) if xs else np.zeros(0, dt))
        parts = gather((cat(c_parts, np.uint32), cat(h_parts, bool), mine, host(oc), host(oh), (o_lo, o_hi),
                        (hi - lo == 0) or ok_dtype))
        if rank == 0:
            r_valid = v if use_valid else None
            (wc, wh), winfo = pipeline.assign_packed(obs, r_valid, whitelist_sorted=wls if use_wl else None,
                                                     true_barcodes=cells[:200].tolist() if use_tb else None, form="u32", **kw)
            gc = np.concatenate([p[0] for p in parts])
            gh = np.concatenate([p[1] for p in parts])
            same = np.array_equal(gc, wc) and np.array_equal(gh, wh.astype(bool))
            infos = all(without_assigned(p[2]) == without_assigned(winfo) for p in parts)
            assigned = sum(p[2]["assigned_reads"] for p in parts) == winfo["assigned_reads"]
            other = all(np.array_equal(p[3], wc[p[5][0]:p[5][1]]) and np.array_equal(p[4], wh[p[5][0]:p[5][1]].astype(bool)) for p in parts)
            record("case %d (t=%d %s)" % (k, t, split), same and infos and assigned and other and all(p[6] for p in parts)
                   and winfo["edges"] > 1000, "same %s infos %s assigned %s other %s: %s vs %s" % (same, infos, assigned, other,
                                                                                            parts[0][2], winfo))


def check_no_valid_row(rank, world, gather, record):
    _, _, obs, valid = dataset(5, 3000, N_CELLS)
    lo, hi = bounds("uneven", world, obs.size)[rank]
    tl = bdist.Tally()
    none = torch.zeros(hi - lo, dtype=torch.bool, device=bd._device())
    tl.add(cuda(obs[lo:hi]), none)
    info = tl.finish(threshold=2, n_cells=10)
    c, h = tl.assign(cuda(obs[lo:hi]), none)
    try:
        tl.assign(cuda(obs[lo:lo + 1]))
        raised = False
    except ValueError:
        raised = True
    tl.free()
    infos = gather(info)
    record("no valid row", raised and not h.any().item() and c.numel() == hi - lo
           and all(i == {"reads": obs.size, "valid_reads": 0} for i in infos))


def check_merged_set(rank, world, gather, record):
    """The read map finish installs equals ops.dedup_reads on the concatenation: a 10^6-read C4-shaped input, several batches per
    rank."""
    wl, cells, obs, valid, cfg = synth.make_dataset("C4", reads=1_000_000)
    lo, hi = bounds("uneven", world, obs.size)[rank]
    tl = bdist.Tally()
    for a, z in batches(lo, hi, 4 + rank, rank):
        tl.add(cuda(obs[a:z], torch.uint32), cuda(valid[a:z], torch.bool))
    T = {}
    info = tl.finish(threshold=2, n_cells=cfg["n_cells"], whitelist_sorted=cuda(np.sort(wl)), timings=T)
    names = ("distinct", "counts", "sorted_pos", "sorted_distinct")
    got = {k: host(getattr(tl._rm, k)).astype(np.int64) for k in names}
    tl.free()
    want = ops.dedup_reads(obs, valid)
    ok = all(np.array_equal(got[k], getattr(want, k).astype(np.int64)) for k in names)
    stages = all(k in T for k in ("exchange_merge", "tally_finish", "edges", "centres", "cluster", "collective_bytes"))
    widths = gather(tl._rm.n_distinct if tl._rm is not None else 0)
    record("merged set", ok and stages and info["distinct"] == want.n_distinct and len(set(widths)) == 1 and want.n_distinct > 100000,
           str(T))


def check_refusals(rank, world, gather, record):
    """A rank-local problem in finish makes every rank raise, and a correct finish works afterwards."""
    _, cells, obs, valid = dataset(11, 30000, N_CELLS)
    lo, hi = bounds("uneven", world, obs.size)[rank]
    kw = dict(threshold=1, n_cells=100)
    want = None
    if rank == 0:
        want = pipeline.assign_packed(obs, valid, form="u32", **kw)
    tl = bdist.Tally()
    tl.add(cuda(obs[lo:hi]), cuda(valid[lo:hi], torch.bool))
    last = rank == world - 1
    results = []
    # a whitelist on the host on the last rank: a bad argument
    try:
        tl.finish(whitelist_sorted=torch.from_numpy(obs[:10].view(np.int32)) if last else None, **kw)
        results.append(False)
    except ValueError:
        results.append(True)
    # different scalar arguments on the last rank
    try:
        tl.finish(threshold=2 if last else 1, n_cells=100)
        results.append(False)
    except ValueError:
        results.append(True)
    # a freed tally on the last rank
    if last:
        tl.free()
    try:
        tl.finish(**kw)
        results.append(False)
    except ValueError:
        results.append(True)
    # a fresh tally on every rank works
    tl.free()
    tl = bdist.Tally()
    tl.add(cuda(obs[lo:hi]), cuda(valid[lo:hi], torch.bool))
    info = tl.finish(**kw)
    c, h = tl.assign(cuda(obs[lo:hi]), cuda(valid[lo:hi], torch.bool))
    try:                                                      # add after finish
        tl.add(cuda(obs[lo:hi]))
        results.append(False)
    except BadgerB200Error as e:
        results.append(e.code == BDG_ERR_ARG)
    info2 = tl.finish(**kw)                                   # a second finish on every rank: the same result
    c2, h2 = tl.assign(cuda(obs[lo:hi]), cuda(valid[lo:hi], torch.bool))
    tl.free()
    parts = gather((host(c), host(h), without_assigned(info), results, torch.equal(c, c2) and torch.equal(h, h2),
                    without_assigned(info2) == without_assigned(info)))
    if rank == 0:
        (wc, wh), winfo = want
        same = np.array_equal(np.concatenate([p[0] for p in parts]), wc) and np.array_equal(np.concatenate([p[1] for p in parts]),
                                                                                           wh.astype(bool))
        record("refusals", same and all(p[2] == without_assigned(winfo) and all(p[3]) and p[4] and p[5] for p in parts),
               str([p[3] for p in parts]))


def check_count_past_32_bits(rank, world, gather, record):
    """Two ranks add 2^31 rows of one barcode each: every rank's count fits 32 bits, the merged one does not."""
    b = torch.full((1 << 28,), 0x1234567, dtype=torch.int32, device=bd._device())
    tl = bdist.Tally()
    for _ in range(8):
        tl.add(b)
    try:
        tl.finish(threshold=1, n_cells=1)
        refused = False
    except BadgerB200Error as e:
        refused = e.code == BDG_ERR_ARG
    tl.free()
    tl = bdist.Tally()
    for _ in range(7):
        tl.add(b)
    tl.add(b[:-1] if rank == world - 1 else b)                # 2^32 - 1 in all: still a uint32 count
    info = tl.finish(threshold=1, n_cells=1, true_barcodes=[0x1234567])
    c, h = tl.assign(b[:5])
    tl.free()
    del b
    ok = info["valid_reads"] == (1 << 32) - 1 and info["distinct"] == 1 and bool(h.all().item()) and bool((c == 0x1234567).all().item())
    record("count past 32 bits", refused and ok, str(info))


def battery(rank, world, gather, which):
    results = []

    def record(name, ok, detail=""):
        results.append((name, bool(ok), detail))
    if which == "count":
        check_count_past_32_bits(rank, world, gather, record)
        return results
    check_cases(rank, world, gather, record)
    check_no_valid_row(rank, world, gather, record)
    check_merged_set(rank, world, gather, record)
    check_refusals(rank, world, gather, record)
    return results


# ---------------------------------------------------------------------------------------------------------------- the worlds
@pytest.mark.parametrize("world", [2, 3])
def test_gloo_world_on_one_gpu(world):
    assert_world(run_world(battery, world, "gloo", "all"), world)


def test_nccl_world_one_gpu_per_rank():
    n = torch.cuda.device_count()
    if n < 2:
        print("skipped: an NCCL world needs two GPUs, this box has %d" % n)
        pytest.skip("an NCCL world needs two GPUs, this box has %d" % n)
    world = min(4, n)
    assert_world(run_world(battery, world, "nccl", "all"), world)


def test_a_merged_count_of_2_32_is_refused_on_every_rank():
    assert_world(run_world(battery, 2, "gloo", "count"), 2)


# ------------------------------------------------------------------------------------ a world of one, in this process
def test_world_of_one_without_a_process_group(claimed_without_group):
    for t, use_wl, use_valid, use_tb, high_sens, order, dtype, _ in CASES:
        wl, cells, obs, valid = dataset(300 + t, N_READS, N_CELLS)
        wls = np.sort(wl)
        kw = dict(threshold=t, n_cells=N_CELLS, high_sens=high_sens, centre_order=order, whitelist_sorted=cuda(wls, dtype) if use_wl else None,
                  true_barcodes=cuda(cells[:200], dtype) if use_tb else None)
        out = []
        for make in (bdist.Tally, bd.Tally):
            tl = make()
            for a, z in batches(0, obs.size, 3, t):
                tl.add(cuda(obs[a:z], dtype), cuda(valid[a:z], torch.bool) if use_valid else None)
            info = tl.finish(**kw)
            c, h = tl.assign(cuda(obs, dtype), cuda(valid, torch.bool) if use_valid else None)
            out.append((c, h, dict(info)))
            tl.free()
        (c, h, info), (wc, wh, winfo) = out
        assert torch.equal(c, wc) and torch.equal(h, wh) and info == winfo


def raw_parts(tallies, dev):
    """The sets of `tallies` (bdg_dev_tally_copy) side by side: (keys int32[P, W], counts int64[P, W], firsts int64[P, W], sizes,
    rows)."""
    L = badger_b200.lib()
    info = []
    for t in tallies:
        n, r, v = C.c_size_t(0), C.c_ulonglong(0), C.c_ulonglong(0)
        assert L.bdg_tally_info(t._handle(), C.byref(n), C.byref(r), C.byref(v)) == BDG_OK
        info.append((int(n.value), int(r.value), int(v.value)))
    W = max(i[0] for i in info)
    keys = torch.zeros((len(tallies), W), dtype=torch.int32, device=dev)
    cnts = torch.zeros((len(tallies), W), dtype=torch.int64, device=dev)
    firsts = torch.zeros((len(tallies), W), dtype=torch.int64, device=dev)
    for p, t in enumerate(tallies):
        assert L.bdg_dev_tally_copy(t._handle(), keys[p].data_ptr(), cnts[p].data_ptr(), firsts[p].data_ptr(), bd._stream()) == BDG_OK
    return keys, cnts, firsts, info


def test_merge_parts_refusals_each_followed_by_a_working_call(claimed_without_group):
    """bdg_dev_tally_merge_parts refuses, leaving the set as it was: a part that is not ascending, an own part that is not the
    handle's set, a wrong size; then the correct call gives the tally of the rank-major concatenation."""
    L, dev = badger_b200.lib(), bd._device()
    _, _, obs, valid = dataset(21, 40000, N_CELLS)
    half = 25000
    ta, tb = bd.Tally(), bd.Tally()
    ta.add(cuda(obs[:10000]), cuda(valid[:10000], torch.bool))
    ta.add(cuda(obs[10000:half]), cuda(valid[10000:half], torch.bool))
    tb.add(cuda(obs[half:]), cuda(valid[half:], torch.bool))
    keys, cnts, firsts, info = raw_parts([ta, tb], dev)
    W = keys.shape[1]
    sizes = [i[0] for i in info]
    rows = [i[1] for i in info]
    total_rows, total_valid = sum(rows), sum(i[2] for i in info)

    def merge(k, c, f, sz, my=0):
        return L.bdg_dev_tally_merge_parts(ta._handle(), k.data_ptr(), c.data_ptr(), f.data_ptr(), (C.c_size_t * 2)(0, W),
                                           (C.c_size_t * 2)(*sz), (C.c_ulonglong * 2)(0, rows[0]), 2, my, total_rows, total_valid,
                                           bd._stream())
    bad = keys.clone()
    bad[1, [3, 4]] = bad[1, [4, 3]]                           # part 1 not ascending
    assert merge(bad, cnts, firsts, sizes) == BDG_ERR_ARG
    bad = cnts.clone()
    bad[0, 7] += 1                                            # own part differs from the handle's set
    assert merge(keys, bad, firsts, sizes) == BDG_ERR_ARG
    assert merge(keys, cnts, firsts, [sizes[0] - 1, sizes[1]]) == BDG_ERR_ARG    # wrong size of the own part
    assert merge(keys, cnts, firsts, sizes, my=1) == BDG_ERR_ARG                # part 1 is not this handle's set
    again = raw_parts([ta], dev)                              # the set is as it was
    assert torch.equal(again[0][0, :sizes[0]], keys[0, :sizes[0]]) and torch.equal(again[1][0, :sizes[0]], cnts[0, :sizes[0]])
    assert merge(keys, cnts, firsts, sizes) == BDG_OK
    assert merge(keys, cnts, firsts, sizes) == BDG_ERR_ARG    # a merged tally takes no second merge
    with pytest.raises(BadgerB200Error):
        ta.add(cuda(obs[:10]))                                # nor a batch
    kw = dict(threshold=2, n_cells=100)
    info_a = ta.finish(**kw)                                  # the one-process finish over the merged set
    ca, ha = ta.assign(cuda(obs), cuda(valid, torch.bool))
    (wc, wh), winfo = pipeline.assign_packed(obs, valid, form="u32", **kw)
    assert np.array_equal(host(ca), wc) and np.array_equal(host(ha), wh.astype(bool))
    assert dict(info_a, reads=obs.size) == winfo              # (device.Tally counts the rows it was given itself)
    ta.free(); tb.free()
    tf = bdist.Tally()                                        # a freed tally refuses finish
    tf.free()
    with pytest.raises(ValueError):
        tf.finish(**kw)


def pcie_probe(out_dir):
    """HtoD + DtoH bytes of one add and one assign of R rows of distributed.Tally (a world of one), at two sizes.  Prints them as
    one JSON line."""
    from torch.profiler import ProfilerActivity, profile
    from test_device_tensors_gpu import memcpy_bytes
    badger_b200.init()
    wl, _, obs, valid = dataset(123, 1000000, N_CELLS)
    d_obs, d_valid = cuda(obs), cuda(valid, torch.bool)
    moved = {}

    def traced(name, fn):
        fn()                                                   # warm: first-use allocations are not per read
        torch.cuda.synchronize()
        out = os.path.join(out_dir, name)
        os.mkdir(out)
        with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        prof.export_chrome_trace(os.path.join(out, "trace.json"))
        moved[name] = memcpy_bytes(out)

    for R in (250000, 1000000):
        t = bdist.Tally()
        traced("add_%d" % R, lambda: t.add(d_obs[:R], d_valid[:R]))
        t.finish(threshold=2, n_cells=600, whitelist_sorted=cuda(np.sort(wl)))
        traced("assign_%d" % R, lambda: t.assign(d_obs[:R], d_valid[:R]))
        t.free()
    print(json.dumps(moved))


def test_only_sizes_cross_pcie_per_add_and_assign(tmp_path):
    """The profiler runs in a process of its own, as in test_batched_step_gpu.py."""
    code = "import sys; sys.path[:0] = %r; import test_distributed_tally_gpu as m; m.pcie_probe(%r)" % ([TESTS, ROOT], str(tmp_path))
    res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stderr[-4000:]
    moved = json.loads(res.stdout.strip().splitlines()[-1])
    print("PCIe bytes:", moved)
    for what in ("add", "assign"):
        assert moved["%s_1000000" % what] < 4096 and moved["%s_250000" % what] < 4096
