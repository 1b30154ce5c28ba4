#!/usr/bin/env python3
"""The correction step in batches (device.Tally) against one call (device.assign_packed), on the C5 config as named: 10⁸ reads,
threshold 2, the 3·10⁶-entry whitelist.  Both forms start from the reads in page-locked host memory and end with the per-read
result there:
  one      the reads are uploaded whole, device.assign_packed runs once, the result comes back;
  batched  pass 1 uploads batch after batch and adds it to a tally, finish runs the stages, pass 2 uploads every batch again and
           assigns it, its result coming back batch by batch (only one batch of reads is on the device at a time).
Each form runs in a process of its own, so that the library's grow-only workspaces of one do not count for the other: one
warm-up step, then --steps timed steps, each ended by a device synchronise.  Peak device memory is the largest
total - free of torch.cuda.mem_get_info, sampled every millisecond over the process (the library allocates outside torch's
allocator), less what was in use before the first step.  The forms alternate --reps times; their results must be equal.

--past-limit also adds the C5 reads K times (K·10⁸ rows, > 2^31) to one tally from device memory, with true_barcodes so that the
centres do not depend on the scale of the counts, and checks that assigning the reads gives the result of a one-batch tally.
Prints one JSON line per run with the card's name and power limit, read in the same run.

    python tools/batched_step_time.py [--batches 10] [--steps 2] [--reps 2] [--past-limit 22] [--out DIR]
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import badger_b200  # noqa: E402
from badger_b200 import synth  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


class PeakMemory:
    """Largest device memory in use (total - free), sampled every millisecond on a thread."""

    def __init__(self, torch):
        self.torch, self.peak, self.stop = torch, 0, False
        self.base = self.used()
        self.th = threading.Thread(target=self.run, daemon=True)
        self.th.start()

    def used(self):
        free, total = self.torch.cuda.mem_get_info()
        return total - free

    def run(self):
        while not self.stop:
            self.peak = max(self.peak, self.used())
            time.sleep(0.001)

    def close(self):
        self.stop = True
        self.th.join()
        return max(self.peak, self.used()) - self.base


def worker(args):
    import torch
    from badger_b200 import device as bd
    badger_b200.init([0])
    dev = bd._device()
    d = np.load(os.path.join(args.data, "c5.npz"))
    obs, valid, wl, cells = d["obs"], d["valid"], d["wl"], d["cells"]
    h_obs = torch.from_numpy(obs.view(np.int32)).pin_memory()
    h_valid = torch.from_numpy(valid).pin_memory()
    R = obs.size
    d_wl = torch.from_numpy(wl.view(np.int32)).to(dev)
    kw = dict(threshold=2, n_cells=10_000, whitelist_sorted=d_wl)
    pts = [R * k // args.batches for k in range(args.batches + 1)]
    torch.cuda.synchronize()
    mem = PeakMemory(torch)
    out_c = torch.empty(R, dtype=torch.int32).pin_memory()
    out_h = torch.empty(R, dtype=torch.bool).pin_memory()
    phases = {}

    def one():
        (c, h), info = bd.assign_packed(h_obs.to(dev, non_blocking=True), h_valid.to(dev, non_blocking=True), **kw)
        out_c.copy_(c, non_blocking=True); out_h.copy_(h, non_blocking=True)
        torch.cuda.synchronize()
        return info

    def batched():
        t = bd.Tally()
        t0 = time.perf_counter()
        for s, e in zip(pts[:-1], pts[1:]):
            t.add(h_obs[s:e].to(dev, non_blocking=True), h_valid[s:e].to(dev, non_blocking=True))
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        info = t.finish(**kw)
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        for s, e in zip(pts[:-1], pts[1:]):
            c, h = t.assign(h_obs[s:e].to(dev, non_blocking=True), h_valid[s:e].to(dev, non_blocking=True))
            out_c[s:e].copy_(c, non_blocking=True); out_h[s:e].copy_(h, non_blocking=True)
        torch.cuda.synchronize()
        t3 = time.perf_counter()
        t.free()
        for k, v in (("add", t1 - t0), ("finish", t2 - t1), ("assign", t3 - t2)):
            phases.setdefault(k, []).append(round(v, 4))
        return info

    run = one if args.form == "one" else batched
    info = run()                                              # warm-up
    phases.clear()
    times = []
    for _ in range(args.steps):
        t0 = time.perf_counter()
        info = run()
        times.append(time.perf_counter() - t0)
    peak = mem.close()
    digest = hashlib.sha256(out_c.numpy().tobytes() + out_h.numpy().tobytes()).hexdigest()[:16]
    rec = dict(form=args.form, reads=R, batches=args.batches if args.form == "batched" else 1, step_s=[round(x, 4) for x in times],
               peak_device_bytes=int(peak), info=info, result_sha256_16=digest)
    if phases:
        rec["phases_s"] = phases
    print(json.dumps(rec))


def past_limit(args):
    """K additions of the C5 reads from device memory, then the per-read result against a one-batch tally."""
    import torch
    from badger_b200 import device as bd
    badger_b200.init([0])
    dev = bd._device()
    d = np.load(os.path.join(args.data, "c5.npz"))
    d_obs = torch.from_numpy(d["obs"].view(np.int32)).to(dev)
    d_valid = torch.from_numpy(d["valid"]).to(dev)
    R, K = d_obs.numel(), args.past_limit
    kw = dict(threshold=2, n_cells=10_000, whitelist_sorted=torch.from_numpy(d["wl"].view(np.int32)).to(dev),
              true_barcodes=torch.from_numpy(d["cells"].view(np.int32)).to(dev))
    ref = bd.Tally()
    ref.add(d_obs, d_valid)
    info1 = ref.finish(**kw)
    want = ref.assign(d_obs, d_valid)
    ref.free()
    torch.cuda.synchronize()
    t = bd.Tally()
    adds = []
    t0 = time.perf_counter()
    for _ in range(K):
        a0 = time.perf_counter()
        t.add(d_obs, d_valid)
        adds.append(time.perf_counter() - a0)
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    info = t.finish(**kw)
    torch.cuda.synchronize()
    t2 = time.perf_counter()
    c, h = t.assign(d_obs, d_valid)
    torch.cuda.synchronize()
    t3 = time.perf_counter()
    same = bool(torch.equal(c, want[0]) and torch.equal(h, want[1]))
    t.free()
    exp = dict(info1, reads=K * R, valid_reads=K * info1["valid_reads"])
    print(json.dumps(dict(form="past_limit", batches=K, rows=K * R, rows_over_2_31=K * R / 2 ** 31, add_total_s=round(t1 - t0, 3),
                          add_median_s=round(float(np.median(adds)), 4), finish_s=round(t2 - t1, 3), assign_one_batch_s=round(t3 - t2, 4),
                          result_equals_one_batch=same, info_equals_scaled=info == exp, info=info)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", type=int, default=10)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--past-limit", type=int, default=22, help="K additions of the 1e8 reads; 0: skip")
    ap.add_argument("--out", default=None, help="also append the JSON lines to DIR/batched_step_time.jsonl")
    ap.add_argument("--form", default=None, help=argparse.SUPPRESS)
    ap.add_argument("--data", default=None, help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.form == "past_limit":
        return past_limit(args)
    if args.form:
        return worker(args)
    gpu = card()
    lines = []
    with tempfile.TemporaryDirectory() as tmp:
        t0 = time.perf_counter()
        wl, cells, obs, valid, _ = synth.make_dataset("C5", workers=os.cpu_count() or 1)
        np.savez(os.path.join(tmp, "c5.npz"), obs=obs, valid=valid, wl=np.sort(wl), cells=cells)
        del obs, valid
        print("C5 generated in %.0f s" % (time.perf_counter() - t0), file=sys.stderr)
        forms = ["one", "batched"] * args.reps + (["past_limit"] if args.past_limit else [])
        for form in forms:
            cmd = [sys.executable, os.path.abspath(__file__), "--form", form, "--data", tmp, "--batches", str(args.batches),
                   "--steps", str(args.steps), "--past-limit", str(args.past_limit)]
            res = subprocess.run(cmd, capture_output=True, text=True)
            if res.returncode:
                sys.stderr.write(res.stderr)
                raise SystemExit("%s run failed" % form)
            rec = json.loads(res.stdout.strip().splitlines()[-1])
            rec["gpu"] = gpu
            lines.append(rec)
            print(json.dumps(rec), flush=True)
    shas = {r["result_sha256_16"] for r in lines if "result_sha256_16" in r}
    infos = {json.dumps(r["info"], sort_keys=True) for r in lines if r["form"] in ("one", "batched")}
    summary = dict(form="summary", equal_results=len(shas) == 1, equal_info=len(infos) == 1, gpu=gpu)
    for f in ("one", "batched"):
        runs = [r for r in lines if r["form"] == f]
        summary[f + "_median_step_s"] = float(np.median([x for r in runs for x in r["step_s"]]))
        summary[f + "_peak_device_gb"] = round(max(r["peak_device_bytes"] for r in runs) / 1e9, 2)
    print(json.dumps(summary))
    lines.append(summary)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "batched_step_time.jsonl"), "a") as fh:
            for r in lines:
                fh.write(json.dumps(r) + "\n")
    if not (summary["equal_results"] and summary["equal_info"]):
        raise SystemExit("the two forms differ")


if __name__ == "__main__":
    main()
