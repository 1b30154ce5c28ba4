#!/usr/bin/env python3
"""The dealing of the join conditions to the devices, measured on ONE device: for nparts in 2, 4, 8 every part is built alone
(device-resident input, CUDA events, best of 3) and the slowest part is what a strong-scaling step on nparts devices would take.
Development tool; bench.py --gpus N is the measurement of record."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import badger_b200  # noqa: E402
from badger_b200 import synth  # noqa: E402


def main():
    badger_b200.init([0])
    L = badger_b200.lib()
    cfg_name = os.environ.get("BAL_CONFIG", "C4")
    wl, cells, obs, valid, cfg = synth.make_dataset(cfg_name, workers=min(32, len(os.sched_getaffinity(0))))
    s = synth.sorted_unique(obs[valid])
    t = int(cfg["threshold"])
    dev = torch.device("cuda", 0)
    n = int(s.size)
    d_sorted = torch.from_numpy(s.view(np.int32)).to(dev)
    cap = 40 * n
    d_a = torch.empty(cap, dtype=torch.int32, device=dev); d_b = torch.empty(cap, dtype=torch.int32, device=dev)
    d_d = torch.empty(cap, dtype=torch.uint8, device=dev); d_c = torch.zeros(1, dtype=torch.int64, device=dev)
    st = torch.cuda.current_stream()

    def go(part, nparts):
        badger_b200._lib.check(L.bdg_dev_edges_build(d_sorted.data_ptr(), n, t, part, nparts, d_a.data_ptr(), d_b.data_ptr(), d_d.data_ptr(),
                                                     cap, d_c.data_ptr(), st.cuda_stream))

    def timed(part, nparts):
        go(part, nparts); torch.cuda.synchronize()
        best = 1e30
        for _ in range(3):
            e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
            e0.record(st); go(part, nparts); e1.record(st); e1.synchronize()
            best = min(best, e0.elapsed_time(e1))
        return best, int(d_c.item())

    if os.environ.get("BAL_ONE"):                    # "part/nparts": that part alone, twice (for an ncu launch list of the second call)
        part, nparts = (int(x) for x in os.environ["BAL_ONE"].split("/"))
        go(part, nparts); torch.cuda.synchronize()
        go(part, nparts); torch.cuda.synchronize()
        print("part %d of %d: %d edges" % (part, nparts, int(d_c.item())))
        return
    whole, edges = timed(0, 1)
    print("%s N=%d t=%d: whole job %.3f ms, %d edges" % (cfg_name, n, t, whole, edges))
    for nparts in (2, 4, 8):
        ms, es = [], []
        for p in range(nparts):
            m, e = timed(p, nparts)
            ms.append(m); es.append(e)
        print("nparts=%d  parts %s  max %.3f ms  sum %.3f ms  efficiency %.3f  edges %s  per part %s" % (
            nparts, " ".join("%.2f" % x for x in ms), max(ms), sum(ms), whole / (nparts * max(ms)),
            "ok" if sum(es) == edges else "MISMATCH %d" % sum(es), " ".join(str(e) for e in es)))


if __name__ == "__main__":
    main()
