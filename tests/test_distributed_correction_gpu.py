"""badger_b200.distributed, the correction step over a process group, against the one-process step on the concatenation of the
ranks' inputs in rank order: the results, concatenated in rank order, and `info` must be equal element for element.

Worlds of 2 and 3 ranks run on gloo with every rank on the first GPU; a world of min(4, GPUs) ranks runs on NCCL with one GPU
per rank.  Each world is one set of spawned processes that runs every check and reports to the test; the reference runs on
rank 0 in the same process as that rank's distributed call, so that centre_order="set" meets the same set order."""
import ctypes as C

import numpy as np
import pytest
import torch

import badger_b200
from badger_b200 import device as bd
from badger_b200 import distributed as bdist
from badger_b200 import ops, pipeline
from gpu_helpers import assert_world, claimed_without_group, cuda, dataset, host, run_world

pytestmark = pytest.mark.gpu

N_READS = 100000
N_CELLS = 300
CASES = [  # threshold, whitelist, valid mask, true barcodes, high_sens, centre_order, barcode dtype, how the reads are split
    (1, True, True, False, False, None, torch.int32, "uneven"),
    (2, False, False, False, False, None, torch.uint32, "first_empty"),
    (2, True, True, False, True, None, torch.int32, "uneven"),
    (2, False, True, True, True, "set", torch.int32, "last_invalid"),
    (3, True, True, False, False, None, torch.uint32, "uneven"),
    (3, False, True, True, False, None, torch.int32, "first_empty"),
]


def bounds(split, world, n):
    """[lo, hi) of every rank: uneven weights 3, 1, 2, 3, 1, 2, ...; "first_empty" gives rank 0 no rows."""
    w = np.array([0 if (split == "first_empty" and r == 0) else (3, 1, 2)[r % 3] for r in range(world)], float)
    if world == 1:
        w[:] = 1
    cut = np.concatenate([[0], np.round(np.cumsum(w) / w.sum() * n)]).astype(int)
    return [(int(cut[r]), int(cut[r + 1])) for r in range(world)]


# ---------------------------------------------------------------------------------------------------------------- the checks
def check_cases(rank, world, gather, record):
    for k, (t, use_wl, use_valid, use_tb, high_sens, order, dtype, split) in enumerate(CASES):
        wl, cells, obs, valid = dataset(900 + k, N_READS, N_CELLS)
        b = bounds(split, world, obs.size)
        v = valid.copy()
        if split == "last_invalid":
            v[b[-1][0]:] = False
        lo, hi = b[rank]
        wls = np.sort(wl)
        kw = dict(threshold=t, n_cells=N_CELLS, high_sens=high_sens, centre_order=order)
        (c, h), info = bdist.assign_packed(cuda(obs[lo:hi], dtype), cuda(v[lo:hi], torch.bool) if use_valid else None,
                                           whitelist_sorted=cuda(wls, dtype) if use_wl else None,
                                           true_barcodes=cuda(cells[:200], dtype) if use_tb else None, **kw)
        ok_dtype = c.dtype == dtype and h.dtype == torch.bool and c.numel() == hi - lo
        parts = gather((host(c), host(h), info, obs[lo:hi], v[lo:hi], ok_dtype))
        if rank == 0:
            r_obs = np.concatenate([p[3] for p in parts])
            r_valid = np.concatenate([p[4] for p in parts])
            (wc, wh), winfo = pipeline.assign_packed(r_obs, r_valid if use_valid else None, whitelist_sorted=wls if use_wl else None,
                                                     true_barcodes=cells[:200].tolist() if use_tb else None, form="u32", **kw)
            gc = np.concatenate([p[0] for p in parts])
            gh = np.concatenate([p[1] for p in parts])
            same = np.array_equal(gc, wc) and np.array_equal(gh, wh.astype(bool)) and all(p[2] == winfo for p in parts)
            record("case %d (t=%d %s)" % (k, t, split), same and all(p[5] for p in parts) and winfo["edges"] > 1000,
                   "info %s vs %s" % (parts[0][2], winfo))


def check_edge_cases(rank, world, gather, record):
    _, _, obs, valid = dataset(5, 3000, N_CELLS)
    lo, hi = bounds("uneven", world, obs.size)[rank]
    (c, h), info = bdist.assign_packed(cuda(obs[lo:hi]), torch.zeros(hi - lo, dtype=torch.bool, device=bd._device()),
                                       threshold=2, n_cells=10)
    infos = gather(info)
    record("all invalid", not h.any().item() and c.numel() == hi - lo and all(i == {"reads": obs.size, "valid_reads": 0} for i in infos))
    (c, h), info = bdist.assign_packed(torch.empty(0, dtype=torch.int32, device=bd._device()), threshold=1, n_cells=10)
    infos = gather(info)
    record("all empty", c.numel() == 0 and all(i == {"reads": 0, "valid_reads": 0} for i in infos))


def check_merge_centres_rounds(rank, world, gather, record):
    wl, cells, obs, valid = dataset(77, 120000, N_CELLS)
    wls = np.sort(wl)
    for split in ("uneven", "first_empty"):
        lo, hi = bounds(split, world, obs.size)[rank]
        rm = bd.dedup_reads(cuda(obs[lo:hi], torch.uint32), cuda(valid[lo:hi], torch.bool))
        merged, n_valid, n_rows = bdist.dedup_merge(rm)
        names = ("distinct", "counts", "sorted_pos", "sorted_distinct")
        got = {k: host(getattr(merged, k)).astype(np.int64) for k in names}
        cen = pipeline.select_centres(merged, N_CELLS, 25, cuda(wls), None, bd.centres_above)
        want = ops.dedup_reads(obs, valid)                                        # (a new dedup: the merged token dies here)
        ok = all(np.array_equal(got[k], getattr(want, k).astype(np.int64)) for k in names)
        record("merge %s" % split, ok and (n_valid, n_rows) == (int(valid.sum()), obs.size) and merged.n_distinct == want.n_distinct)
        all_cen = gather(list(cen))
        want_cen = pipeline.select_centres(want, N_CELLS, 25, wls, None)
        record("centres %s" % split, all(c == list(want_cen) for c in all_cen) and len(want_cen) > 100)

    s_np = np.unique(obs[valid])
    s = cuda(s_np)
    a, b, _ = bd.edges(s, 2, part=rank, nparts=world)
    centres = np.asarray(list(dict.fromkeys(cells[:250].tolist())), np.uint32)
    ci, lv = bdist.cluster_levels(s, a, b, centres)
    lv = host(lv).copy()
    lv[lv == ops.LEVEL_HAS_EDGE] = ops.LEVEL_NONE
    parts = gather((host(a), host(b), host(ci).view(np.int32), lv))
    ua = np.concatenate([p[0] for p in parts]); ub = np.concatenate([p[1] for p in parts])
    want_ci, want_lv = ops.cluster_levels(s_np, ua, ub, centres, 2)
    same = all(np.array_equal(p[2], want_ci) and np.array_equal(p[3], want_lv) for p in parts)
    record("rounds", same and (want_ci >= 0).sum() > len(centres) and (world == 1 or max(p[0].size for p in parts) < ua.size))


def battery(rank, world, gather):
    results = []

    def record(name, ok, detail=""):
        results.append((name, bool(ok), detail))
    check_cases(rank, world, gather, record)
    check_edge_cases(rank, world, gather, record)
    check_merge_centres_rounds(rank, world, gather, record)
    return results


# ---------------------------------------------------------------------------------------------------------------- the worlds
@pytest.mark.parametrize("world", [2, 3])
def test_gloo_world_on_one_gpu(world):
    assert_world(run_world(battery, world, "gloo", timeout=1200), world)


def test_nccl_world_one_gpu_per_rank():
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("an NCCL world needs two GPUs")
    world = min(4, n)
    assert_world(run_world(battery, world, "nccl", timeout=1200), world)


# ------------------------------------------------------------------------------------ a world of one, in this process
def test_world_of_one_without_a_process_group(claimed_without_group):
    for t, use_wl, use_valid, use_tb, high_sens, order, dtype, _ in CASES[2:5]:
        wl, cells, obs, valid = dataset(300 + t, N_READS, N_CELLS)
        wls = np.sort(wl)
        args = (cuda(obs, dtype), cuda(valid, torch.bool) if use_valid else None)
        kw = dict(threshold=t, n_cells=N_CELLS, high_sens=high_sens, centre_order=order, whitelist_sorted=cuda(wls, dtype) if use_wl else None,
                  true_barcodes=cuda(cells[:200], dtype) if use_tb else None)
        T = {}
        (c, h), info = bdist.assign_packed(*args, timings=T, **kw)
        (wc, wh), winfo = bd.assign_packed(*args, **kw)
        assert torch.equal(c, wc) and torch.equal(h, wh) and info == winfo
        assert T["collective_bytes"]["lists"] == 12 * info["distinct"] and T["gather"] > 0


def test_argument_errors_leave_it_usable(claimed_without_group):
    _, _, obs, valid = dataset(3, 20000, N_CELLS)
    d_obs, d_valid = cuda(obs), cuda(valid, torch.bool)
    kw = dict(threshold=1, n_cells=100)
    with pytest.raises(ValueError):
        bdist.assign_packed(torch.from_numpy(obs.view(np.int32)), **kw)                 # CPU tensor
    with pytest.raises(TypeError):
        bdist.assign_packed(d_obs.to(torch.int64), **kw)                                # wrong dtype
    with pytest.raises(TypeError):
        bdist.assign_packed(d_obs, d_valid.to(torch.float32), **kw)
    with pytest.raises(ValueError):
        bdist.assign_packed(d_obs, whitelist_sorted=torch.from_numpy(obs.view(np.int32)), **kw)
    # the merge refuses a stale token and a list that is not the token's own
    L, dev = badger_b200.lib(), bd._device()
    old = bd.dedup_reads(d_obs)
    lists = bdist._lists(old, dev)
    n = old.n_distinct
    new = bd.dedup_reads(d_obs, d_valid)

    def merge(tok, lst, size):
        base = lst.data_ptr()
        nd, mt = C.c_size_t(0), C.c_ulonglong(0)
        return L.bdg_dev_dedup_merge(tok, base, base + 4 * lst.shape[1], base + 8 * lst.shape[1], (C.c_size_t * 1)(0),
                                     (C.c_size_t * 1)(size), 1, 0, C.byref(nd), C.byref(mt), bd._stream())
    assert merge(old.token, lists, n) == badger_b200._lib.BDG_ERR_ARG                   # stale token
    other = bdist._lists(new, dev)
    wrong = other.clone()
    wrong[0, -1] += 1                                                                   # (the largest barcode, still ascending)
    assert merge(new.token, wrong, new.n_distinct) == badger_b200._lib.BDG_ERR_ARG       # not the token's list
    assert merge(new.token, other, new.n_distinct - 1) == badger_b200._lib.BDG_ERR_ARG   # not its size
    assert merge(new.token, other, new.n_distinct) == badger_b200._lib.BDG_OK
    (c, h), info = bdist.assign_packed(d_obs, d_valid, **kw)
    (wc, wh), winfo = bd.assign_packed(d_obs, d_valid, **kw)
    assert torch.equal(c, wc) and torch.equal(h, wh) and info == winfo
