"""badger_b200.distributed, the correction step over a process group, against the one-process step on the concatenation of the
ranks' inputs in rank order: the results, concatenated in rank order, and `info` must be equal element for element.

Worlds of 2 and 3 ranks run on gloo with every rank on the first GPU; a world of min(4, GPUs) ranks runs on NCCL with one GPU
per rank.  Each world is one set of spawned processes that runs every check and reports to the test; the reference runs on
rank 0 in the same process as that rank's distributed call, so that centre_order="set" meets the same set order."""
import ctypes as C
import os
import queue
import socket
import sys
import time
import traceback

import numpy as np
import pytest
import torch

import badger_b200
from badger_b200 import device as bd
from badger_b200 import distributed as bdist
from badger_b200 import ops, pipeline, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
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


def dataset(seed, n_reads=N_READS, n_cells=N_CELLS, err=0.08):
    rng = synth.rng_for(seed)
    wl = synth.make_whitelist(20000, rng)
    cells = synth.pick_cells(wl, n_cells, rng)
    obs, valid = synth.simulate_reads(cells, n_reads, err, rng)
    return wl, cells, obs, valid


def cuda(a, dtype=torch.int32):
    """A numpy barcode array (uint32 bits kept) or mask as a tensor on the first claimed device."""
    if dtype in (torch.bool, torch.uint8):
        return torch.from_numpy(np.ascontiguousarray(a)).to(bd._device()).to(dtype)
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.uint32).view(np.int32)).to(bd._device()).view(dtype)


def host(t):
    t = t.cpu()
    return t.view(torch.int32).numpy().view(np.uint32) if t.dtype in (torch.int32, torch.uint32) else t.numpy()


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
        wl, cells, obs, valid = dataset(900 + k)
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
    _, _, obs, valid = dataset(5, 3000)
    lo, hi = bounds("uneven", world, obs.size)[rank]
    (c, h), info = bdist.assign_packed(cuda(obs[lo:hi]), torch.zeros(hi - lo, dtype=torch.bool, device=bd._device()),
                                       threshold=2, n_cells=10)
    infos = gather(info)
    record("all invalid", not h.any().item() and c.numel() == hi - lo and all(i == {"reads": obs.size, "valid_reads": 0} for i in infos))
    (c, h), info = bdist.assign_packed(torch.empty(0, dtype=torch.int32, device=bd._device()), threshold=1, n_cells=10)
    infos = gather(info)
    record("all empty", c.numel() == 0 and all(i == {"reads": 0, "valid_reads": 0} for i in infos))


def check_merge_centres_rounds(rank, world, gather, record):
    wl, cells, obs, valid = dataset(77, 120000)
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
def _worker(rank, world, backend, port, q):
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    try:
        os.environ["MASTER_ADDR"] = "127.0.0.1"
        os.environ["MASTER_PORT"] = str(port)
        dev = rank if backend == "nccl" else 0
        torch.cuda.set_device(dev)
        dist.init_process_group(backend, rank=rank, world_size=world)
        badger_b200.init([dev])

        def gather(obj):
            out = [None] * world
            dist.all_gather_object(out, obj)
            return out
        q.put((rank, battery(rank, world, gather)))
        dist.barrier()
        dist.destroy_process_group()
    except BaseException:
        q.put((rank, [("rank %d raised" % rank, False, traceback.format_exc())]))


def run_world(world, backend, timeout=1200):
    import torch.multiprocessing as mp
    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        port = sk.getsockname()[1]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, world, backend, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    deadline = time.monotonic() + timeout
    got = {}
    try:
        while len(got) < world:
            rank, res = q.get(timeout=max(1.0, deadline - time.monotonic()))
            got[rank] = res
            if any(not ok for _, ok, _ in res):
                break                      # a failed rank may leave the others waiting in a collective
    except queue.Empty:
        pass
    finally:
        for p in procs:
            p.join(max(1.0, min(120.0, deadline - time.monotonic())))
        for p in procs:
            if p.is_alive():
                p.terminate()
                p.join(30)
            if p.is_alive():
                p.kill()
                p.join()
    return got


def assert_world(got, world):
    failed = [(r, name, detail) for r, res in sorted(got.items()) for name, ok, detail in res if not ok]
    assert not failed, failed
    assert sorted(got) == list(range(world)), "ranks that did not report: %s" % sorted(set(range(world)) - set(got))
    print({r: len(res) for r, res in got.items()})


@pytest.mark.parametrize("world", [2, 3])
def test_gloo_world_on_one_gpu(world):
    assert_world(run_world(world, "gloo"), world)


def test_nccl_world_one_gpu_per_rank():
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("an NCCL world needs two GPUs")
    world = min(4, n)
    assert_world(run_world(world, "nccl"), world)


# ------------------------------------------------------------------------------------ a world of one, in this process
@pytest.fixture
def claimed():
    import torch.distributed as dist
    assert not dist.is_initialized()
    assert badger_b200.init([0]) == 1
    yield
    badger_b200.init()


def test_world_of_one_without_a_process_group(claimed):
    for t, use_wl, use_valid, use_tb, high_sens, order, dtype, _ in CASES[2:5]:
        wl, cells, obs, valid = dataset(300 + t)
        wls = np.sort(wl)
        args = (cuda(obs, dtype), cuda(valid, torch.bool) if use_valid else None)
        kw = dict(threshold=t, n_cells=N_CELLS, high_sens=high_sens, centre_order=order, whitelist_sorted=cuda(wls, dtype) if use_wl else None,
                  true_barcodes=cuda(cells[:200], dtype) if use_tb else None)
        T = {}
        (c, h), info = bdist.assign_packed(*args, timings=T, **kw)
        (wc, wh), winfo = bd.assign_packed(*args, **kw)
        assert torch.equal(c, wc) and torch.equal(h, wh) and info == winfo
        assert T["collective_bytes"]["lists"] == 12 * info["distinct"] and T["gather"] > 0


def test_argument_errors_leave_it_usable(claimed):
    _, _, obs, valid = dataset(3, 20000)
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
