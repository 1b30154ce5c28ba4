#!/usr/bin/env python3
"""Drop-in for algbio/Badger's badger.py (reference badger.py:23-175): same options, same TSV in/out, with the
barcode graph built by the B200 kernels (badger_b200).  `barcodes.py` is the README's name for this script.

Differences, all outside the hot path (SURVEY.md §2): FASTQ/FASTA/BAM input needs the extraction step
(ssw / pysam / Biopython), which is out of scope - pass the extraction TSV; --stats is not provided.
"""
import argparse
import logging
import sys
from io import StringIO
from traceback import print_exc

import numpy as np
import pandas as pd

from badger_b200 import BarcodeGraph, init

logger = logging.getLogger('BarcodeGraph')

# reference: extract_raw_barcodes.py:33-34 (+ the README's spellings, README.md:112-113,137-138)
BARCODE_CALLING_MODES = {'tenX_v2': 16, 'tenX_v3': 16, '10x': 16, 'visium': 16}


def parse_args(args):
    parser = argparse.ArgumentParser(formatter_class=argparse.RawDescriptionHelpFormatter)
    parser.add_argument("--barcodes", "-b", help="(README spelling) tsv file containing the observed cell barcodes; "
                        "same as --reads", type=str, dest="bar_file", default=None)
    parser.add_argument("--threshold", "-t", help="Maximal accepted difference between barcodes "
                        "(1 runs the sorted search, 2 and 3 the joined searches on multi-block seeds; >= 4 runs the dense all-pairs kernel, meant for small inputs)",
                        type=int, dest="threshold", default=1)
    parser.add_argument("--reads", "-r", help="TSV from barcode extraction",
                        type=str, dest="reads", default=None)
    parser.add_argument("--ground_truth", help="File connecting each observed barcode to its read ID containing true barcode, only used for statistics "
                        "(accepted for compatibility; the statistics it feeds are outside this drop-in: a warning is logged and the file is not read)",
                        type=str, default=None)
    parser.add_argument("--barcode_list", "-l", help="List of all possible barcodes for the used method, helps identify correct barcodes",
                        type=str, dest="barcode_list", default=None)
    parser.add_argument("--data_type", "-d", help="Type of single cell sequencing data in the input",
                        choices=BARCODE_CALLING_MODES.keys(), type=str)
    parser.add_argument("--true_barcodes", help="List of all true barcodes of the input data, for example obtained from short read data",
                        type=str, default=None)
    parser.add_argument("--n_cells", "-c", help="expected number of cell associated barcodes",
                        type=int, default=5000)
    parser.add_argument("--output", "-o", help="File prefix for output files",
                        type=str, default="OUT")
    parser.add_argument("--interval", "-i", help="Percentage by which the number of cells is allowed to differ from estimated cell number, default 25%%", default=25, type=int)
    parser.add_argument("--stats", "-s", action='store_true', help="(not provided by the B200 path)", default=False)
    parser.add_argument("--threads", "-tr", dest="threads", default=1, type=int)
    parser.add_argument("--high_sens", "-hs", action='store_true', help="if set, Badger is run in high sensitivity mode. This increases recall but decreases precision. "
                        "Ties between equally near centres are broken by the iteration order of a Python set of strings, in the reference and here alike: "
                        "the result is reproducible only under a fixed PYTHONHASHSEED", default=False)
    parser.add_argument("--devices", help="comma-separated CUDA device ids (default: all visible)", type=str, default=None)
    parser.add_argument("--no_native_io", action='store_true', default=False,
                        help="read and write the TSVs through pandas and the dict-shaped BarcodeGraph (the slower route the native "
                             "reader falls back to by itself when it declines a file)")
    ns = parser.parse_args(args)
    if ns.reads is None:
        ns.reads = ns.bar_file
    if ns.reads is None:
        parser.error("the following arguments are required: --reads/-r")
    return ns


def set_logger(logger_instance):
    logger_instance.setLevel(logging.INFO)
    c_handler = logging.StreamHandler(stream=sys.stdout)
    c_handler.setLevel(logging.INFO)
    c_handler.setFormatter(logging.Formatter('%(asctime)s - %(levelname)s - %(message)s'))
    logger_instance.addHandler(c_handler)
    logger_instance.info("Starting")


def run_native(args, bc_len, true_barcodes):
    """The same run without per-read Python: extraction TSV and whitelist read by the native library (badger_b200.tsvio),
    barcodes packed on the GPU, the array form of graph construction / clustering / assignment
    (badger_b200.pipeline.assign_packed), output TSV written by the native library.  Same output file and same stdout as
    the route below.  Returns False - nothing done yet - when the reader declines the file (anything pandas would treat
    specially): the caller then goes through pandas like the reference."""
    from badger_b200 import ops, pipeline, tsvio
    from badger_b200.common import rank
    try:
        tsv = tsvio.ExtractionTsv(args.reads, bc_len)
    except tsvio.Unsupported as e:
        logger.info("%s - reading through pandas", e)
        return False
    with tsv:
        logger.info("Imported barcodes from file")
        init([int(x) for x in args.devices.split(",")] if args.devices else None)
        logger.info("Initializing Graph")
        print("k:", 6)                                          # index.py:21 (QGramIndex.__init__)
        has = tsv.has_barcode
        ranks = np.zeros(tsv.rows, np.uint32)
        packed, ok = ops.pack16(tsv.seqs16[has])
        if not ok.all():                                        # common.py:24: rank() raises KeyError(letter)
            bad = bytes(tsv.seqs16[has][int(np.argmin(ok))]).decode("ascii", "replace")
            raise KeyError(next(c for c in bad if c not in "ACGT"))
        ranks[has] = packed
        whitelist = None
        if args.barcode_list:                                   # badger.py:82-88
            whitelist = ops.pack16_sorted(tsvio.whitelist_records(args.barcode_list))     # packed, sorted, distinct: on the device
        tb = [rank(bc, bc_len) for bc in true_barcodes] if true_barcodes else None
        (centre, has_centre), info = pipeline.assign_packed(ranks, has, threshold=args.threshold, n_cells=args.n_cells, interval=args.interval,
                                                            whitelist_sorted=whitelist, true_barcodes=tb, high_sens=args.high_sens,
                                                            centre_order="set", form="u32")
        logger.info("Graph construction done")
        print(1)                                                # barcode_graph.py:289 prints the round number
        print(2)
        logger.info("Clustering done")
        tsv.write32(args.output + "_output_file.tsv", centre, has_centre)
        print(info["disconnected"])                             # badger.py:131-132
    return True


def main(args):
    args = parse_args(args)
    set_logger(logger)
    if args.data_type is None or args.data_type not in BARCODE_CALLING_MODES:
        logger.error("Please specify the type of single cell data used. Options are tenX_v2, tenX_v3 (aliases 10x, visium).")
        exit(-3)
    bc_len = BARCODE_CALLING_MODES[args.data_type]
    if args.ground_truth:
        logger.warning("--ground_truth only feeds the reference's accuracy statistics (badger.py:146-174), which this drop-in does not compute: ignored")
    true_barcodes = args.true_barcodes
    if true_barcodes:                                           # badger.py:74-80
        true_barcodes = pd.read_csv(true_barcodes, sep="\t", header=None)
        true_barcodes = true_barcodes.iloc[:, 0].tolist()
        if true_barcodes[0][-1] == '1':
            for i in range(len(true_barcodes)):
                true_barcodes[i] = true_barcodes[i][:-2]
        true_barcodes = set(true_barcodes)

    out = args.output
    if args.reads.endswith("tsv") and not args.stats and not args.no_native_io:
        if run_native(args, bc_len, true_barcodes):
            return

    if args.barcode_list:                                       # badger.py:82-88
        with open(args.barcode_list, "r") as list_file:
            barcode_list = set(list_file.read().split("\n"))
    else:
        barcode_list = None

    if not args.reads.endswith("tsv"):
        logger.error("FASTQ/FASTA/BAM input needs the barcode extraction step, which this drop-in does not replace; "
                     "run the reference's extract_raw_barcodes.py and pass its TSV")
        exit(-3)
    reads = pd.read_csv(args.reads, sep="\t")                   # badger.py:91-111
    ids = reads["#read_id"].tolist()
    observed = reads["barcode"].fillna('*').tolist()
    read_assignment = []
    barcodes = reads["barcode"].dropna()
    barcodes = barcodes[barcodes != "*"]
    barcodes = barcodes[barcodes != "barcode"]
    barcodes = barcodes.tolist()
    for i in range(len(ids)):
        if ids[i] != "#read_id":
            o = observed[i]
            if o != "barcode":
                if len(o) == bc_len + 1:
                    o = o[:-1]
                read_assignment.append((ids[i], o))
    logger.info("Imported barcodes from file")

    init([int(x) for x in args.devices.split(",")] if args.devices else None)
    logger.info("Initializing Graph")
    graph = BarcodeGraph(args.threshold)
    graph.graph_construction(barcodes, bc_len, args.threads)
    logger.info("Graph construction done")

    if not args.stats:
        graph.cluster(true_barcodes, barcode_list, args.n_cells, bc_len, args.interval)
        logger.info("Clustering done")
        graph.output_file(read_assignment, out, true_barcodes, bc_len, args.high_sens)

    disconnected = len(graph.counts.keys()) - len(graph.edges.keys())     # badger.py:131-132
    print(disconnected)

    if args.stats:
        logger.error("--stats (thesis statistics, reference stats.py) is outside this drop-in's scope")
        exit(-3)


def cli(argv=None):
    """The command's top level (reference badger.py:177-196): any failure is logged as 'Barcode Graph failed' and exits with -1.
    badger.py and its README alias barcodes.py both enter here."""
    try:
        main(sys.argv[1:] if argv is None else argv)
    except SystemExit:
        raise
    except KeyboardInterrupt:
        raise
    except:  # noqa: E722 - same top-level behaviour as the reference (badger.py:177-196)
        if logger.handlers:
            strout = StringIO()
            print_exc(file=strout)
            s = strout.getvalue()
            if s:
                logger.critical("Barcode Graph failed" + s)
            else:
                print_exc()
        else:
            sys.stderr.write("Barcode Graph failed")
            print_exc()
        sys.exit(-1)


if __name__ == "__main__":
    cli()
