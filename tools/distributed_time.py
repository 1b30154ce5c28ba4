#!/usr/bin/env python3
"""The correction step over one process per GPU (badger_b200.distributed.assign_packed) against one process holding all the
GPUs (badger_b200.device.assign_packed), on the same seeded reads, alternating the two forms after a warm-up of each.

    torchrun --nproc_per_node P tools/distributed_time.py [--configs C4] [--reps 3] [--one-process-gpus 8] [--backend nccl]

Rank r runs on GPU r mod (visible GPUs): with fewer GPUs than ranks, --backend gloo lets ranks share a GPU (a check of the results
at full size; its times are not those of one GPU per rank).  Rank r takes the r-th contiguous slice of the reads (rank 0
generates them once and shares them through a temporary directory).  The one-process form runs in a helper process that rank 0 starts, so that both forms keep their workspaces warm; while one form
runs the other processes wait on a gloo (CPU) barrier.  Every stage of the distributed form ends in a device synchronise; a
stage's time is the largest over the ranks.  The per-read results of the two forms are compared byte for byte on every rank.
Rank 0 prints one JSON line per config with the card's name and power limit."""
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


def one_process(conn, n_gpus, tmp, kw):
    """Helper: device.assign_packed on all reads with n_gpus claimed; answers "run" (seconds) and "save" (writes the result)."""
    import torch
    import badger_b200
    from badger_b200 import device as bd
    badger_b200.init(list(range(n_gpus)))
    obs, valid, wls = (np.load(os.path.join(tmp, f)) for f in ("obs.npy", "valid.npy", "wl.npy"))
    d_obs = torch.from_numpy(obs.view(np.int32)).cuda(0)
    d_valid = torch.from_numpy(valid).cuda(0)
    d_wl = torch.from_numpy(wls.view(np.int32)).cuda(0)
    out = None
    while True:
        cmd = conn.recv()
        if cmd == "run":
            for g in range(n_gpus):
                torch.cuda.synchronize(g)
            t0 = time.perf_counter()
            out = bd.assign_packed(d_obs, d_valid, whitelist_sorted=d_wl, **kw)
            for g in range(n_gpus):
                torch.cuda.synchronize(g)
            conn.send(time.perf_counter() - t0)
        elif cmd == "save":
            (c, h), info = out
            np.save(os.path.join(tmp, "one_centre.npy"), c.cpu().numpy())
            np.save(os.path.join(tmp, "one_has.npy"), h.cpu().numpy())
            conn.send(info)
        else:
            conn.send(None)
            return


def bounds(world, n):
    cut = [n * r // world for r in range(world + 1)]
    return [(cut[r], cut[r + 1]) for r in range(world)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="C4")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--one-process-gpus", type=int, default=8)
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
    n_one = min(args.one_process_gpus, torch.cuda.device_count())
    for name in args.configs.split(","):
        cfg = synth.CONFIGS[name]
        kw = dict(threshold=cfg["threshold"], n_cells=cfg["n_cells"])
        box = [None]
        if rank == 0:
            tmp = tempfile.mkdtemp(prefix="bdg_dist_")
            wl, _, obs, valid, _ = synth.make_dataset(name, workers=os.cpu_count() or 1)
            np.save(os.path.join(tmp, "obs.npy"), obs)
            np.save(os.path.join(tmp, "valid.npy"), valid)
            np.save(os.path.join(tmp, "wl.npy"), np.sort(wl))
            del obs, valid, wl
            box = [tmp]
            ctx = mp.get_context("spawn")
            here, there = ctx.Pipe()
            helper = ctx.Process(target=one_process, args=(there, n_one, tmp, kw))
            helper.start()
        dist.broadcast_object_list(box, src=0, group=cpu)
        tmp = box[0]
        obs = np.load(os.path.join(tmp, "obs.npy"), mmap_mode="r")
        lo, hi = bounds(world, obs.size)[rank]
        d_obs = torch.from_numpy(np.array(obs[lo:hi]).view(np.int32)).cuda(dev)
        d_valid = torch.from_numpy(np.array(np.load(os.path.join(tmp, "valid.npy"), mmap_mode="r")[lo:hi])).cuda(dev)
        d_wl = torch.from_numpy(np.load(os.path.join(tmp, "wl.npy")).view(np.int32)).cuda(dev)

        def distributed(timings=None):
            torch.cuda.synchronize(dev)
            dist.barrier(group=cpu)
            t0 = time.perf_counter()
            out = bdist.assign_packed(d_obs, d_valid, whitelist_sorted=d_wl, timings=timings, **kw)
            torch.cuda.synchronize(dev)
            return out, time.perf_counter() - t0

        def single():
            dist.barrier(group=cpu)
            s = None
            if rank == 0:
                here.send("run")
                s = here.recv()
            dist.barrier(group=cpu)
            return s

        (c, h), info = distributed()[0]                               # warm both forms
        single()
        same = True
        if rank == 0:
            here.send("save")
            one_info = here.recv()
            same = info == one_info
        dist.barrier(group=cpu)
        one_c = np.load(os.path.join(tmp, "one_centre.npy"), mmap_mode="r")[lo:hi]
        one_h = np.load(os.path.join(tmp, "one_has.npy"), mmap_mode="r")[lo:hi]
        mine = c.cpu().numpy()
        same = (same and mine.tobytes() == np.ascontiguousarray(one_c).tobytes()
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
            print(json.dumps({"config": name, "reads": int(obs.size), "ranks": world, "backend": args.backend,
                              "rank_gpus": min(world, torch.cuda.device_count()), "one_process_gpus": n_one, "gpu": gpu,
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
