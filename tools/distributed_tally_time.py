#!/usr/bin/env python3
"""The batched correction step over one process per GPU (badger_b200.distributed.Tally) against the one-process tally
(badger_b200.device.Tally) on the rank-major concatenation of the same batches, on the same seeded reads.

    torchrun --nproc_per_node P tools/distributed_tally_time.py [--configs C4,C5] [--batches 4] [--reps 3] [--backend nccl]

Rank r runs on GPU r mod (visible GPUs): with fewer GPUs than ranks, --backend gloo lets ranks share a GPU (a check of the results
at full size; its times are not those of one GPU per rank).  Rank r takes the r-th contiguous slice of the reads and adds it in
--batches uneven batches; the one-process tally adds every rank's batches in rank order, in a helper process that rank 0 starts
on rank 0's GPU (while one form runs, the other processes wait on a gloo barrier).  Every stage ends in a device synchronise; a
stage's time is the largest over the ranks.  The per-read results of the two forms are compared byte for byte on every rank, and
`info` too.  Rank 0 prints one JSON line per config with the card's name and power limit."""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def bounds(world, n):
    cut = [n * r // world for r in range(world + 1)]
    return [(cut[r], cut[r + 1]) for r in range(world)]


def batch_cuts(lo, hi, k, seed):
    """[lo, hi) in k uneven batches (sizes between 1/2 and 3/2 of the mean)."""
    w = np.random.default_rng(seed).uniform(0.5, 1.5, k)
    cut = lo + np.round(np.cumsum(np.concatenate([[0], w])) / w.sum() * (hi - lo)).astype(np.int64)
    return [(int(a), int(b)) for a, b in zip(cut[:-1], cut[1:])]


def rank_major(world, n, k):
    return [c for r, (lo, hi) in enumerate(bounds(world, n)) for c in batch_cuts(lo, hi, k, r)]


def one_process(conn, dev, tmp, kw, world, k):
    """Helper: device.Tally over every rank's batches in rank order; answers "run" (seconds) and "save" (writes the result)."""
    import torch
    import badger_b200
    from badger_b200 import device as bd
    torch.cuda.set_device(dev)
    badger_b200.init([dev])
    obs, valid, wls = (np.load(os.path.join(tmp, f)) for f in ("obs.npy", "valid.npy", "wl.npy"))
    d_obs = torch.from_numpy(obs.view(np.int32)).cuda(dev)
    d_valid = torch.from_numpy(valid).cuda(dev)
    d_wl = torch.from_numpy(wls.view(np.int32)).cuda(dev)
    cuts = rank_major(world, obs.size, k)
    out = None
    while True:
        cmd = conn.recv()
        if cmd == "run":
            torch.cuda.synchronize(dev)
            t0 = time.perf_counter()
            t = bd.Tally()
            for a, z in cuts:
                t.add(d_obs[a:z], d_valid[a:z])
            info = t.finish(whitelist_sorted=d_wl, **kw)
            c, h = t.assign(d_obs, d_valid)
            torch.cuda.synchronize(dev)
            out = (c, h, dict(info))
            t.free()
            conn.send(time.perf_counter() - t0)
        elif cmd == "save":
            c, h, info = out
            np.save(os.path.join(tmp, "one_centre.npy"), c.cpu().numpy())
            np.save(os.path.join(tmp, "one_has.npy"), h.cpu().numpy())
            conn.send(info)
        else:
            conn.send(None)
            return


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="C4")
    ap.add_argument("--batches", type=int, default=4, help="batches per rank")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--backend", default="nccl", choices=["nccl", "gloo"])
    args = ap.parse_args()
    import torch
    import torch.distributed as dist
    import torch.multiprocessing as mp
    import badger_b200
    from badger_b200 import distributed as bdist
    from badger_b200 import synth
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    dev = int(os.environ.get("LOCAL_RANK", rank)) % torch.cuda.device_count()
    torch.cuda.set_device(dev)
    dist.init_process_group(args.backend)
    cpu = dist.new_group(backend="gloo")
    badger_b200.init([dev])
    gpu = card() if rank == 0 else None
    for name in args.configs.split(","):
        cfg = synth.CONFIGS[name]
        kw = dict(threshold=cfg["threshold"], n_cells=cfg["n_cells"])
        box = [None]
        if rank == 0:
            tmp = tempfile.mkdtemp(prefix="bdg_dtally_")
            wl, _, obs, valid, _ = synth.make_dataset(name, workers=os.cpu_count() or 1)
            np.save(os.path.join(tmp, "obs.npy"), obs)
            np.save(os.path.join(tmp, "valid.npy"), valid)
            np.save(os.path.join(tmp, "wl.npy"), np.sort(wl))
            del obs, valid, wl
            box = [tmp]
            ctx = mp.get_context("spawn")
            here, there = ctx.Pipe()
            helper = ctx.Process(target=one_process, args=(there, dev, tmp, kw, world, args.batches))
            helper.start()
        dist.broadcast_object_list(box, src=0, group=cpu)
        tmp = box[0]
        obs = np.load(os.path.join(tmp, "obs.npy"), mmap_mode="r")
        lo, hi = bounds(world, obs.size)[rank]
        d_obs = torch.from_numpy(np.array(obs[lo:hi]).view(np.int32)).cuda(dev)
        d_valid = torch.from_numpy(np.array(np.load(os.path.join(tmp, "valid.npy"), mmap_mode="r")[lo:hi])).cuda(dev)
        d_wl = torch.from_numpy(np.load(os.path.join(tmp, "wl.npy")).view(np.int32)).cuda(dev)
        cuts = [(a - lo, z - lo) for a, z in batch_cuts(lo, hi, args.batches, rank)]

        def distributed(T):
            torch.cuda.synchronize(dev)
            dist.barrier(group=cpu)
            t0 = time.perf_counter()
            t = bdist.Tally()
            for a, z in cuts:
                t.add(d_obs[a:z], d_valid[a:z])
            torch.cuda.synchronize(dev)
            T["add"] = time.perf_counter() - t0
            info = t.finish(whitelist_sorted=d_wl, timings=T, **kw)
            t1 = time.perf_counter()
            c, h = t.assign(d_obs, d_valid)
            torch.cuda.synchronize(dev)
            T["assign"] = time.perf_counter() - t1
            out = (c, h, dict(info))
            t.free()
            return out, time.perf_counter() - t0

        def single():
            dist.barrier(group=cpu)
            s = None
            if rank == 0:
                here.send("run")
                s = here.recv()
            dist.barrier(group=cpu)
            return s

        (c, h, info), _ = distributed({})                             # warm both forms
        single()
        infos = [None] * world
        dist.all_gather_object(infos, info, group=cpu)
        same = True
        if rank == 0:
            here.send("save")
            one_info = here.recv()
            drop = (lambda i: {k: v for k, v in i.items() if k != "assigned_reads"})
            same = (all(drop(i) == drop(one_info) for i in infos)
                    and sum(i.get("assigned_reads", 0) for i in infos) == one_info.get("assigned_reads", 0))
        dist.barrier(group=cpu)
        one_c = np.load(os.path.join(tmp, "one_centre.npy"), mmap_mode="r")[lo:hi]
        one_h = np.load(os.path.join(tmp, "one_has.npy"), mmap_mode="r")[lo:hi]
        same = (same and c.cpu().numpy().tobytes() == np.ascontiguousarray(one_c).tobytes()
                and h.cpu().numpy().tobytes() == np.ascontiguousarray(one_h).tobytes())
        flag = torch.tensor([0 if same else 1], dtype=torch.int32)
        dist.all_reduce(flag, op=dist.ReduceOp.MAX, group=cpu)
        del c, h
        times = {"distributed": [], "one_process": []}
        stages, traffic = [], None
        for _ in range(args.reps):
            T = {}
            _, t = distributed(T)
            traffic = T.pop("collective_bytes")
            per_rank = [None] * world
            dist.all_gather_object(per_rank, (t, T), group=cpu)
            times["distributed"].append(max(x[0] for x in per_rank))
            stages.append({k: max(x[1].get(k, 0.0) for x in per_rank) for k in per_rank[0][1]})
            times["one_process"].append(single())
        if rank == 0:
            med = {k: round(float(np.median([s[k] for s in stages])), 4) for k in stages[0]}
            print(json.dumps({"config": name, "reads": int(obs.size), "ranks": world, "batches_per_rank": args.batches,
                              "backend": args.backend, "rank_gpus": min(world, torch.cuda.device_count()),
                              "one_gpu_per_rank": world <= torch.cuda.device_count(), "one_process_gpus": 1, "gpu": gpu,
                              "same_result": bool(flag.item() == 0), "info": info,
                              "distributed_s": [round(x, 4) for x in times["distributed"]],
                              "one_process_s": [round(x, 4) for x in times["one_process"]],
                              "distributed_median_s": round(float(np.median(times["distributed"])), 4),
                              "one_process_median_s": round(float(np.median(times["one_process"])), 4),
                              "distributed_stage_median_s": med, "collective_bytes_rank0": traffic}), flush=True)
            here.send("stop")
            here.recv()
            helper.join()
        del d_obs, d_valid, d_wl, obs
        dist.barrier(group=cpu)
        if rank == 0:
            shutil.rmtree(tmp, ignore_errors=True)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
