"""What the GPU tests share: the claiming fixtures, the simulated data set, numpy <-> tensor conversion, and the harness that runs a
battery of checks in a world of spawned processes, one rank each."""
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
from badger_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture
def claimed():
    assert badger_b200.init() >= 1
    yield
    badger_b200.init()


@pytest.fixture
def claimed_without_group():
    """A world of one in this process: the first GPU only, no process group."""
    import torch.distributed as dist
    assert not dist.is_initialized()
    assert badger_b200.init([0]) == 1
    yield
    badger_b200.init()


def dataset(seed, n_reads, n_cells=600, err=0.08):
    """(whitelist sorted, cells, read barcodes, valid mask) of a simulated run over a 20000-barcode whitelist."""
    rng = synth.rng_for(seed)
    wl = synth.make_whitelist(20000, rng)
    cells = synth.pick_cells(wl, n_cells, rng)
    obs, valid = synth.simulate_reads(cells, n_reads, err, rng)
    return np.sort(wl), cells, obs, valid


def cuda(a, dtype=torch.int32):
    """A numpy barcode array (uint32 bits kept), mask or byte array as a tensor on the first claimed device."""
    if dtype in (torch.bool, torch.uint8):
        return torch.from_numpy(np.ascontiguousarray(a)).to(bd._device()).to(dtype)
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.uint32).view(np.int32)).to(bd._device()).view(dtype)


def host(t):
    """A barcode tensor as uint32 numpy (the same bits), any other tensor as numpy of its own dtype."""
    t = t.cpu()
    return t.view(torch.int32).numpy().view(np.uint32) if t.dtype in (torch.int32, torch.uint32) else t.numpy()


# ---------------------------------------------------------------------------------------------------------------- the worlds
def _worker(rank, world, backend, port, q, battery, args):
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
        q.put((rank, battery(rank, world, gather, *args)))
        dist.barrier()
        dist.destroy_process_group()
    except BaseException:
        q.put((rank, [("rank %d raised" % rank, False, traceback.format_exc())]))


def run_world(battery, world, backend, *args, timeout=1500):
    """battery(rank, world, gather, *args) -> [(name, ok, detail)] on every rank of a spawned world (gloo: every rank on the first
    GPU; nccl: one GPU per rank); gather(obj) is the list of every rank's obj.  Returns {rank: its list} of the ranks that
    reported."""
    import torch.multiprocessing as mp
    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        port = sk.getsockname()[1]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, world, backend, port, q, battery, args)) for r in range(world)]
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
    print({r: [name for name, _, _ in res] for r, res in got.items()})
