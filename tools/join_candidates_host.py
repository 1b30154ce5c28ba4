#!/usr/bin/env python3
"""Candidates, close pairs and edges of the t = 2 join, counted on the host with the kernel's own per-pair functions.

Buckets the distinct barcodes of a BASELINE config (C4 by default, synthesised as bench.py does) by every join key and runs
every bucket pair through both filters of the join: the three-diagonal quick test with the flag table (the form before the
side filter) and the one-sided filter with the side-aware hand-over (join2_quick, seed_lut_build_sides, bdg_seed.cuh).
The two edge counts must be equal, and the new candidate count is what the kernel's own counter (bench.py
roofline.work.candidates) should show.  Compiles tools/join_candidates_host.cpp with g++ -fopenmp into a temporary directory.

  python3 tools/join_candidates_host.py [--config C4] [--blocks 3,3,3,3,3] [--input sorted.u32]
"""
from __future__ import annotations

import argparse
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

COLS = ["pairs", "cand_old", "cand_new", "near_old", "near_new", "edges_old", "edges_new"]


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--config", default="C4")
    ap.add_argument("--reads", type=int, default=None, help="override the read count of the config")
    ap.add_argument("--blocks", default="3,3,3,3,3", help="bases per block of the t = 2 scheme (BDG_JOIN_BLOCKS)")
    ap.add_argument("--input", default=None, help="sorted distinct barcodes as raw uint32 instead of a synthesised config")
    ap.add_argument("--per-condition", action="store_true")
    args = ap.parse_args()
    with tempfile.TemporaryDirectory() as tmp:
        src = args.input
        if src is None:
            from badger_b200 import synth
            cfg = dict(synth.CONFIGS[args.config])
            if args.reads is not None:
                cfg["reads"] = args.reads
            workers = max(2, min(32, len(os.sched_getaffinity(0))))      # the stream bench.py draws (synth.simulate_reads)
            _, _, obs, valid, _ = synth.make_dataset(cfg, workers=workers)
            src = os.path.join(tmp, "s.u32")
            synth.sorted_unique(obs[valid]).astype("<u4").tofile(src)
        exe = os.path.join(tmp, "join_candidates_host")
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fopenmp", "-I", os.path.join(ROOT, "badger_b200", "csrc"),
                               os.path.join(ROOT, "tools", "join_candidates_host.cpp"), "-o", exe])
        out = subprocess.run([exe, src] + args.blocks.split(","), check=True, capture_output=True, text=True).stdout
    rows = {}
    for line in out.splitlines():
        w = line.split()
        if w[0] == "total":
            rows[w[1]] = np.array([int(x) for x in w[2:]], np.int64)
        elif w[0] == "N":
            n = int(w[1])
        elif args.per_condition:
            print(line)
    print("N = %d distinct barcodes, blocks %s" % (n, args.blocks))
    print("%-10s %14s %14s %14s %8s %14s %14s %12s %12s" % ("", "bucket pairs", "cand (3 diag)", "cand (sides)", "change",
                                                           "D<=2 (3 diag)", "D<=2 (sides)", "edges (3 diag)", "edges (sides)"))
    for g in ("symmetric", "shifted", "all"):
        r = dict(zip(COLS, rows[g]))
        print("%-10s %14d %14d %14d %7.1f%% %14d %14d %12d %12d" % (g, r["pairs"], r["cand_old"], r["cand_new"],
                                                                   100.0 * (r["cand_new"] / max(1, r["cand_old"]) - 1), r["near_old"],
                                                                   r["near_new"], r["edges_old"], r["edges_new"]))
    r = dict(zip(COLS, rows["all"]))
    if r["edges_old"] != r["edges_new"]:
        sys.exit("edge counts differ: %d with the three-diagonal test, %d with the side filter" % (r["edges_old"], r["edges_new"]))


if __name__ == "__main__":
    main()
