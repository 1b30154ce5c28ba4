#!/usr/bin/env python3
"""Lane use of the t = 2 join kernel at C4 (or BAL_CONFIG): one edge construction on one device with a build that counts
(make -C badger_b200/csrc -B EXTRA=-DBDG_JOIN_LANE_STATS), then the counters of bdg_join_lane_stats as one JSON line:
push rounds against hits pushed, candidate batches through the exact distance, and batches through the hand-over check with
the pairs they carry.  `handover_batches_per_close_batch_form` is what the hand-over check ran on while it followed the distance
in the same batch (every batch holding a pair at D <= 2).  Development tool; the counters slow the kernel, so time nothing here."""
import ctypes as C
import json
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
    v = (C.c_ulonglong * 8)()
    badger_b200._lib.check(L.bdg_join_lane_stats(v, 1))          # fails unless the build counts
    badger_b200._lib.check(L.bdg_dev_edges_build(d_sorted.data_ptr(), n, t, 0, 1, d_a.data_ptr(), d_b.data_ptr(), d_d.data_ptr(),
                                                 cap, d_c.data_ptr(), st.cuda_stream))
    torch.cuda.synchronize()
    badger_b200._lib.check(L.bdg_join_lane_stats(v, 1))
    raw = (C.c_ulonglong * 8)()
    badger_b200._lib.check(L.bdg_dev_edges_stats_raw(raw, st.cuda_stream))
    c = [int(x) for x in v]
    rec = dict(config=cfg_name, N=n, t=t, edges=int(d_c.item()),
               push_rounds=c[0], hits_pushed=c[1], push_lane_use=c[1] / max(1, 32 * c[0]),
               dist_batches=c[2], dist_lanes=c[3], dist_lane_use=c[3] / max(1, 32 * c[2]),
               handover_batches_per_close_batch_form=c[4], handover_batches=c[5], handover_lanes=c[6],
               handover_lane_use=c[6] / max(1, 32 * c[5]),
               candidates=int(raw[3]), candidates_within_t=int(raw[6]), owned=int(raw[7]))
    print(json.dumps(rec), flush=True)


if __name__ == "__main__":
    main()
