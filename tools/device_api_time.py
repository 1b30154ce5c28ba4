#!/usr/bin/env python3
"""Host arrays against CUDA tensors for the whole correction step: pipeline.assign_packed(form="u32") (per-read arrays cross
PCIe both ways) against badger_b200.device.assign_packed (they stay on the GPU), on the same seeded config, alternating the two
forms in one process.  Prints one JSON line per config with the card's name and power limit beside the times.

    python tools/device_api_time.py [--configs C4,C5] [--reps 3]
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
from badger_b200 import pipeline, synth  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="C4,C5")
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    import torch
    from badger_b200 import device as bd
    badger_b200.init([0])
    gpu = card()
    for name in args.configs.split(","):
        wl, _, obs, valid, cfg = synth.make_dataset(name, workers=os.cpu_count() or 1)
        wls = np.sort(wl)
        kw = dict(threshold=cfg["threshold"], n_cells=cfg["n_cells"])
        d_obs = torch.from_numpy(obs.view(np.int32)).cuda()
        d_valid = torch.from_numpy(valid).cuda()
        d_wl = torch.from_numpy(wls.view(np.int32)).cuda()

        def host_form():
            return pipeline.assign_packed(obs, valid, whitelist_sorted=wls, form="u32", **kw)

        def device_form():
            out = bd.assign_packed(d_obs, d_valid, whitelist_sorted=d_wl, **kw)
            torch.cuda.synchronize()
            return out

        (hc, hh), hinfo = host_form()                   # warm both, and check that they agree
        (dc, dh), dinfo = device_form()
        same = hinfo == dinfo and np.array_equal(dc.cpu().numpy().view(np.uint32), hc) and np.array_equal(dh.cpu().numpy(), hh.astype(bool))
        times = {"host": [], "device": []}
        for _ in range(args.reps):
            for form, fn in (("host", host_form), ("device", device_form)):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                fn()
                times[form].append(time.perf_counter() - t0)
        print(json.dumps({"config": name, "reads": int(obs.size), "gpu": gpu, "same_result": bool(same),
                          "host_s": [round(x, 4) for x in times["host"]], "device_s": [round(x, 4) for x in times["device"]],
                          "host_median_s": round(float(np.median(times["host"])), 4),
                          "device_median_s": round(float(np.median(times["device"])), 4)}), flush=True)
        del d_obs, d_valid, d_wl


if __name__ == "__main__":
    main()
