#!/usr/bin/env python3
"""Host arrays against CUDA tensors for the whitelist operators: ops.KmerIndex.query / ops.nearest_bounded / ops.member_sorted
(queries uploaded, every result brought back over PCIe) against their badger_b200.device forms (everything stays on the GPU).
Inputs: the C2 config's 3·10⁶-entry whitelist, its observed reads as queries and its 10⁴ cells as nearest targets.  Every case is
warmed up once in each form; the two results must be equal (hits compared after sorting by (query, string), on the GPU), then the
forms alternate for --reps timed calls, each ended by a device synchronise.  Prints one JSON line per case with the card's name and
power limit, read in the same run.

    python tools/device_whitelist_time.py [--reps 3] [--cases kmer4096,kmer65536,kmer1000000,nearest,member]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import badger_b200  # noqa: E402
from badger_b200 import ops, synth  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--cases", default="kmer4096,kmer65536,kmer1000000,nearest,member")
    args = ap.parse_args()
    import torch
    from badger_b200 import device as bd
    badger_b200.init([0])
    gpu = card()
    wl, cells, obs, valid, _ = synth.make_dataset("C2", reads=1_100_000)
    reads = obs[valid]
    dev = bd._device()

    def cuda(a):
        return torch.from_numpy(np.ascontiguousarray(a, dtype=np.uint32).view(np.int32)).to(dev)

    def sorted_hits(hq, hw, cnt, pos):
        """(query, string) keys ascending, with cnt and pos in that order; all on the GPU."""
        if isinstance(hq, np.ndarray):
            hq, hw, cnt, pos = cuda(hq), cuda(hw), torch.from_numpy(cnt).to(dev), torch.from_numpy(np.ascontiguousarray(pos)).to(dev)
        key = (hq.to(torch.int64) << 32) | (hw.to(torch.int64) & 0xFFFFFFFF)
        key, o = torch.sort(key)
        return key, cnt[o], pos[o]

    def same_hits(a, b):
        x, y = sorted_hits(*a), sorted_hits(*b)
        return all(torch.equal(u, v) for u, v in zip(x, y))

    def same_arrays(d, h):
        return all(np.array_equal(x.cpu().numpy(), y) for x, y in zip(d, h))

    d_wl = cuda(wl)
    wls = np.sort(wl)
    d_wls = cuda(wls)
    for case in args.cases.split(","):
        if case.startswith("kmer"):
            Q = int(case[4:])
            q = np.resize(reads, Q)
            d_q = cuda(q)
            hix, dix = ops.KmerIndex(wl), bd.KmerIndex(d_wl)
            host_form = lambda: hix.query(q, min_kmers=4)                      # noqa: E731
            device_form = lambda: dix.query(d_q, min_kmers=4)                  # noqa: E731
            h, d = host_form(), device_form()
            torch.cuda.synchronize()
            same, hits = same_hits(d, h), int(h[0].size)
            del h, d
            row = {"case": "kmer_index_query", "queries": Q, "whitelist": int(wl.size), "min_kmers": 4, "hits": hits}
        elif case == "nearest":
            q = reads[:400_000]
            d_q, d_t = cuda(q), cuda(cells)
            host_form = lambda: ops.nearest_bounded(q, cells, 2)               # noqa: E731
            device_form = lambda: bd.nearest_bounded(d_q, d_t, 2)              # noqa: E731
            h, d = host_form(), device_form()
            same = same_arrays(d, h)
            row = {"case": "nearest_bounded", "queries": int(q.size), "targets": int(cells.size), "max_d": 2,
                   "within_max_d": int((h[0] >= 0).sum())}
        elif case == "member":
            q = np.resize(reads, 1_000_000)
            d_q = cuda(q)
            host_form = lambda: ops.member_sorted(wls, q)                      # noqa: E731
            device_form = lambda: bd.member_sorted(d_wls, d_q)                 # noqa: E731
            h, d = host_form(), device_form()
            same = bool(np.array_equal(d.cpu().numpy(), h))
            row = {"case": "member_sorted", "queries": int(q.size), "whitelist": int(wls.size), "hits": int(h.sum())}
        else:
            raise SystemExit("unknown case %r" % case)
        times = {"host": [], "device": []}
        kernel_ms = []
        for _ in range(args.reps):
            for form, fn in (("host", host_form), ("device", device_form)):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                out = fn()
                torch.cuda.synchronize()
                times[form].append(time.perf_counter() - t0)
                if form == "device" and case.startswith("kmer"):
                    kernel_ms.append(round(dix.info()["kernel_ms"], 3))
                del out
        if case.startswith("kmer"):
            row["device_kernel_ms"] = kernel_ms
            hix.free(); dix.free()
        row.update({"gpu": gpu, "same_result": bool(same), "host_s": [round(x, 4) for x in times["host"]],
                    "device_s": [round(x, 4) for x in times["device"]], "host_median_s": round(float(np.median(times["host"])), 4),
                    "device_median_s": round(float(np.median(times["device"])), 4)})
        print(json.dumps(row), flush=True)


if __name__ == "__main__":
    main()
