"""Edge construction at t = 3 on one GPU: the join form (bdg_join.cuh) against the dense all-pairs kernel.

Random subsets of the C4 set (the C4 synthetic data, 4.57e6 distinct barcodes) at growing sizes, both forms while the dense one
finishes in seconds, then the join alone up to the full set.  Per size and form: device time per step (CUDA events around
bdg_dev_edges_build on torch's stream, L2 overwritten between steps), edges, and the join's counters (work units, pairs tested,
candidates, candidates with D <= 3, owned pairs).  Where both forms run, their edge sets must be equal.
One JSON line per measurement on stdout, appended to --out as well when given.

  python tools/t3_time.py [--dense 25000,50000,100000,200000] [--join 25000,50000,100000,200000,1000000,full] [--steps 3]
Environment: BDG_JOIN3_BLOCKS picks the layout (read once per process)."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import badger_b200  # noqa: E402
from badger_b200 import synth  # noqa: E402


def gpu_label():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except Exception as e:  # noqa: BLE001
        return "unknown (%s)" % e


def run(torch, L, s, mode, steps, flush):
    badger_b200._lib.check(L.bdg_set_edge_mode(mode))
    dev = torch.device("cuda:0")
    stream = torch.cuda.current_stream()
    d_s = torch.from_numpy(s.view(np.int32)).to(dev)
    cap = max(1 << 16, 64 * s.size)
    cnt = torch.zeros(1, dtype=torch.int64, device=dev)
    while True:
        d_a = torch.empty(cap, dtype=torch.int32, device=dev); d_b = torch.empty(cap, dtype=torch.int32, device=dev)
        d_d = torch.empty(cap, dtype=torch.uint8, device=dev)

        def launch():
            badger_b200._lib.check(L.bdg_dev_edges_build(d_s.data_ptr(), s.size, 3, 0, 1, d_a.data_ptr(), d_b.data_ptr(), d_d.data_ptr(), cap,
                                                         cnt.data_ptr(), stream.cuda_stream))
        launch()
        torch.cuda.synchronize()
        n = int(cnt.item())
        if n <= cap:
            break
        cap = n + 1024
    times = []
    for _ in range(steps):
        flush.fill_(1)
        e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
        e0.record(stream); launch(); e1.record(stream); e1.synchronize()
        times.append(e0.elapsed_time(e1))
    raw = (C.c_ulonglong * 8)()
    badger_b200._lib.check(L.bdg_dev_edges_stats_raw(raw, stream.cuda_stream))
    n = int(cnt.item())
    a = d_a[:n].cpu().numpy().view(np.uint32); b = d_b[:n].cpu().numpy().view(np.uint32); d = d_d[:n].cpu().numpy()
    o = np.lexsort((b, a))
    badger_b200._lib.check(L.bdg_set_edge_mode(-1))
    return dict(ms=min(times), ms_all=[round(t, 3) for t in times], edges=n, raw=[int(x) for x in raw]), (a[o], b[o], d[o])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--dense", default="25000,50000,100000,200000")
    ap.add_argument("--join", default="25000,50000,100000,200000,1000000,full")
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    import torch
    os.environ["BDG_JOIN3_MIN_N"] = "0"
    assert badger_b200.init([0]) == 1
    L = badger_b200.lib()
    label = gpu_label()
    workers = min(32, len(os.sched_getaffinity(0)))
    _, _, obs, valid, _ = synth.make_dataset("C4", workers=workers)
    full = synth.sorted_unique(obs[valid])
    del obs, valid
    rng = np.random.default_rng(7)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda:0")
    dense_sizes = [int(x) for x in args.dense.split(",") if x]
    join_sizes = [full.size if x == "full" else int(x) for x in args.join.split(",") if x]
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
    with open(args.out or os.devnull, "a") as fh:
        for n in sorted(set(dense_sizes) | set(join_sizes)):
            s = full if n >= full.size else np.sort(rng.choice(full, n, replace=False)).astype(np.uint32)
            res = {}
            for form, mode in (("dense", 0), ("join", 2)):
                if (form == "dense" and n not in dense_sizes) or (form == "join" and n not in join_sizes):
                    continue
                r, edges = run(torch, L, s, mode, args.steps, flush)
                res[form] = edges
                rec = dict(form=form, N=int(s.size), t=3, ms=round(r["ms"], 3), ms_all=r["ms_all"], edges=r["edges"],
                           layout=os.environ.get("BDG_JOIN3_BLOCKS", "3,2,2,2,2,2,2"), gpu=label)
                if form == "join":
                    raw = r["raw"]
                    rec.update(units=raw[0], pairs_tested=raw[2], candidates=raw[3], cand_d_le3=raw[6], owned=raw[7],
                               warp_busy_ms_sum=raw[4] / 1e6, warp_busy_ms_max=raw[5] / 1e6)
                line = json.dumps(rec)
                print(line, flush=True)
                fh.write(line + "\n")
            if len(res) == 2:
                same = all(np.array_equal(x, y) for x, y in zip(res["dense"], res["join"]))
                print(json.dumps(dict(N=int(s.size), dense_equals_join=same)), flush=True)
                fh.write(json.dumps(dict(N=int(s.size), dense_equals_join=same)) + "\n")
                assert same, "join and dense edge sets differ at N = %d" % s.size


if __name__ == "__main__":
    main()
