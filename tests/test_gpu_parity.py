"""Parity tests proper: the CUDA path, called through the C ABI (badger_b200.ops -> libbadger_b200.so), against
the golden fixtures of the unmodified reference and against the CPU oracle on seeded inputs.
Bit-exact: all of this path is integer work."""
import ctypes as C
import hashlib
import os

import numpy as np
import pytest

import badger_b200
from badger_b200 import BarcodeGraph, KmerIndexer, QGramIndex, ops, synth
from badger_b200.parallel import part_pairs, part_rows
from oracle import oracle as orc

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module", autouse=True)
def _init():
    n = badger_b200.init()
    assert n >= 1
    yield


MODES = {"dense": 0, "sparse": 1, "join": 2}


@pytest.fixture(params=["sparse", "dense", "join"])
def mode(request):
    """Every search strategy of the edge construction (include/badger_b200.h bdg_set_edge_mode) must give the
    reference's edge set.  The join form exists for t = 2 and t = 3: asked for at another threshold, the library takes
    the sparse / dense route, and the edge set must still be the reference's."""
    L = badger_b200.lib()
    badger_b200._lib.check(L.bdg_set_edge_mode(MODES[request.param]))
    yield request.param
    badger_b200._lib.check(L.bdg_set_edge_mode(-1))


def edge_rows(a, b, d):
    a, b, d = ops.canonical(a, b, d)
    return np.stack([a, b, d], 1).astype(np.int64)


def clustered_set(seed, n_cells, reads, perr):
    rng = synth.rng_for(seed)
    cells = rng.integers(0, 1 << 32, n_cells, dtype=np.uint64).astype(np.uint32)
    obs, _ = synth.simulate_reads(cells, reads, perr, rng)
    return np.unique(obs)


# ------------------------------------------------------------------------------------------ golden fixtures
def test_pack16_and_pairs(gold_pairs):
    strs = [p["a"] for p in gold_pairs["pairs"]] + [p["b"] for p in gold_pairs["pairs"]]
    r, v = ops.pack16(strs)
    assert v.all()
    assert r.tolist() == [p["ra"] for p in gold_pairs["pairs"]] + [p["rb"] for p in gold_pairs["pairs"]]
    r2, v2 = ops.pack16(["ACGTACGTACGTACGN", "acgtacgtacgtacgt", "ACGTACGTACGTACGT", "ACGTACGTACGTAC\nT"])
    assert v2.tolist() == [False, False, True, False] and int(r2[2]) == 3840206052
    arr = np.frombuffer("".join(strs).encode(), np.uint8).reshape(-1, 16)         # the record matrix of badger_b200.tsvio
    r3, v3 = ops.pack16(arr)
    assert np.array_equal(r3, r) and v3.all()
    r4, v4 = ops.pack16(arr[::2])                                                   # a strided view is made contiguous first
    assert np.array_equal(r4, r[::2]) and v4.all()
    # every golden pair as a two-node graph: edge iff S >= T(t) and D <= t, stored distance D
    for t in (0, 1, 2, 3, 4):
        for p in gold_pairs["pairs"][::3]:
            s = np.sort(np.asarray([p["ra"], p["rb"]], np.uint32))
            a, b, d = ops.edges_build(s, t)
            want = p["S"] >= orc.T(t) and p["D"] <= t
            assert (a.size == 1) == want, (p, t)
            if want:
                assert int(d[0]) == p["D"] and (int(a[0]), int(b[0])) == (int(s[0]), int(s[1]))


def test_graphs_golden(gold_graphs):
    for g in gold_graphs:
        bg = BarcodeGraph(g["t"])
        bg.graph_construction(g["reads"], 16, 1)
        assert [(k, v) for k, v in bg.counts.items()] == [tuple(x) for x in g["counts"]], g["name"]
        a, b, d = bg.edge_arrays()
        assert np.stack([a, b, d], 1).astype(np.int64).tolist() == g["edges"], g["name"]
        for gc in g["get_close"]:
            assert sorted(bg.index.get_close(orc.unrank(gc["query"]), gc["query"])) == gc["close"]


def test_pipeline_golden(gold_pipeline, tmp_path, capsys):
    import importlib.util
    import logging
    spec = importlib.util.spec_from_file_location("badger_cli", os.path.join(ROOT, "badger.py"))
    cli = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(cli)
    g = gold_pipeline
    # both routes of the CLI: native reader / array pipeline / native writer (default) and pandas + dict-shaped BarcodeGraph
    for k, route in enumerate(([], ["--no_native_io"])):
        out = str(tmp_path / ("OUT%d" % k))
        cli.main(["-r", g["dir"] + "/reads.tsv", "-l", g["dir"] + "/whitelist.txt", "-d", "tenX_v3", "-t", str(g["t"]),
                  "--n_cells", str(g["n_cells"]), "-i", str(g["interval"]), "-o", out] + route)
        for h in list(logging.getLogger("BarcodeGraph").handlers):
            logging.getLogger("BarcodeGraph").removeHandler(h)
        with open(out + "_output_file.tsv", "rb") as fh, open(g["dir"] + "/expected_output_file.tsv", "rb") as ref:
            assert fh.read() == ref.read(), route
        text = capsys.readouterr().out
        assert "reading through pandas" not in text
        tail = [ln for ln in text.splitlines() if ln.strip().lstrip("-").isdigit()]
        assert tail == g["stdout_tail"], route
    # --high_sens: the two routes meet the same set order inside one process
    outs = []
    for k, route in enumerate(([], ["--no_native_io"])):
        out = str(tmp_path / ("HS%d" % k))
        cli.main(["-r", g["dir"] + "/reads.tsv", "-l", g["dir"] + "/whitelist.txt", "-d", "10x", "-t", str(g["t"]), "-hs",
                  "--n_cells", str(g["n_cells"]), "-i", str(g["interval"]), "-o", out] + route)
        for h in list(logging.getLogger("BarcodeGraph").handlers):
            logging.getLogger("BarcodeGraph").removeHandler(h)
        outs.append((open(out + "_output_file.tsv", "rb").read(),
                     [ln for ln in capsys.readouterr().out.splitlines() if ln.strip().lstrip("-").isdigit()]))
    assert outs[0] == outs[1]
    # internals + --high_sens with the centre order the reference iterated
    import pandas as pd
    df = pd.read_csv(g["dir"] + "/reads.tsv", sep="\t")
    bcs = df["barcode"].dropna()
    bcs = bcs[(bcs != "*") & (bcs != "barcode")].tolist()
    bg = BarcodeGraph(g["t"])
    bg.graph_construction(bcs, 16, 1)
    a, b, d = bg.edge_arrays()
    assert np.stack([a, b, d], 1).astype(np.int64).tolist() == g["edges"]
    with open(g["dir"] + "/whitelist.txt") as fh:
        wl = set(fh.read().split("\n"))
    assert bg.get_cluster_centers(None, 16, wl, g["n_cells"], g["interval"]) == g["centres"]
    bg.cluster(None, wl, g["n_cells"], 16, g["interval"])
    assert {k: tuple(v) for k, v in bg.clustering.items()} == {k: (c, l) for k, c, l in g["clustering"]}
    assign = bg.assign_by_cluster(16)
    assert dict(assign) == g["assignments"]
    hs = bg.postprocessing(assign, 16, _centre_order=g["hs_centre_order"])
    assert {k: v for k, v in hs.items() if v not in ("", "*")} == g["hs_assignments"]


def test_packed_pipeline_golden(gold_pipeline):
    """Array form of the whole correction step (badger_b200.pipeline.assign_packed: dedup, edges, centres, clustering rounds
    and the per-read gather all on the GPU operators) against the output TSV of the unmodified reference."""
    import pandas as pd
    from badger_b200 import pipeline
    g = gold_pipeline
    df = pd.read_csv(g["dir"] + "/reads.tsv", sep="\t")
    obs = df["barcode"].fillna("*").tolist()
    emitted = [i != "#read_id" and o != "barcode" for i, o in zip(df["#read_id"].tolist(), obs)]     # badger.py:103-110
    keep = [o[:-1] if len(o) == 17 else o for o in obs]
    valid = np.asarray([len(o) == 16 and not (set(o) - set("ACGT")) for o in keep])
    ranks = np.zeros(len(keep), np.uint32)
    ranks[valid] = synth.rank_many([o for o, v in zip(keep, valid) if v])
    with open(g["dir"] + "/whitelist.txt") as fh:
        wl = [w for w in fh.read().split("\n") if len(w) == 16]
    out, info = pipeline.assign_packed(ranks, valid, threshold=g["t"], n_cells=g["n_cells"], interval=g["interval"],
                                       whitelist_sorted=np.sort(synth.rank_many(wl)))
    want = pd.read_csv(g["dir"] + "/expected_output_file.tsv", sep="\t")["barcode"].tolist()
    got = ["*" if c == pipeline.NONE else orc.unrank(int(c)) for c, e in zip(out.tolist(), emitted) if e]
    assert got == want
    assert info["edges"] == len(g["edges"]) and info["centres"] == len(g["centres"])
    # --high_sens with the centre order the reference iterated
    out_hs, _ = pipeline.assign_packed(ranks, valid, threshold=g["t"], n_cells=g["n_cells"], interval=g["interval"],
                                       whitelist_sorted=np.sort(synth.rank_many(wl)), high_sens=True,
                                       centre_order=[orc.rank(c) for c in g["hs_centre_order"]])
    want_hs = dict(g["hs_assignments"])
    for o, v, c in zip(keep, valid, out_hs.tolist()):
        if v:
            assert (orc.unrank(int(c)) if c != pipeline.NONE else None) == want_hs.get(o), o


def test_packed_pipeline_edge_cases_and_true_barcodes():
    """assign_packed on empty / all-invalid input, and the --true_barcodes branch against the string mirror."""
    from badger_b200 import pipeline
    out, info = pipeline.assign_packed(np.empty(0, np.uint32), threshold=1, n_cells=10)
    assert out.size == 0 and info["reads"] == 0
    out, info = pipeline.assign_packed(np.arange(5, dtype=np.uint32), np.zeros(5, bool), threshold=1, n_cells=10)
    assert (out == pipeline.NONE).all() and info["valid_reads"] == 0
    rng = synth.rng_for(77)
    cells = rng.integers(0, 1 << 32, 50, dtype=np.uint64).astype(np.uint32)
    obs, valid = synth.simulate_reads(cells, 8000, 0.06, rng)
    tb = cells[:40].tolist()
    out, info = pipeline.assign_packed(obs, valid, threshold=2, n_cells=40, true_barcodes=tb, high_sens=True)
    strs = [s.decode() for s in synth.unrank_many(obs[valid]).tolist()]
    bg = BarcodeGraph(2)
    bg.graph_construction(strs, 16, 1)
    bg.cluster([orc.unrank(int(c)) for c in tb], None, 40, 16, 25)
    assign = bg.assign_by_cluster(16)
    used = sorted({orc.rank(v) for v in assign.values() if v not in ("", "*")})
    assign = bg.postprocessing(assign, 16, _centre_order=[orc.unrank(u) for u in used])     # ascending order, as assign_packed's default
    want = [assign[s_] if assign[s_] not in ("", "*") else None for s_ in strs]
    got = [orc.unrank(int(c)) if c != pipeline.NONE else None for c in out[valid].tolist()]
    assert got == want and sum(g is not None for g in got) > 6000


def test_c1_golden(gold_c1):
    wl, cells, obs, valid, cfg = synth.make_dataset("C1")
    strs = [s.decode() for s in synth.unrank_many(obs[valid]).tolist()]
    bg = BarcodeGraph(cfg["threshold"])
    bg.graph_construction(strs, 16, 1)
    assert len(bg.counts) == gold_c1["n_distinct"]
    pairs = np.asarray(list(bg.counts.items()), dtype=np.uint64)
    assert hashlib.sha256(pairs.tobytes()).hexdigest() == gold_c1["counts_sha256"]
    a, b, d = bg.edge_arrays()
    assert np.stack([a, b, d], 1).astype(np.int64).tolist() == gold_c1["edges"]
    wl_set = set(s.decode() for s in synth.unrank_many(wl).tolist()) | {""}
    centres = bg.get_cluster_centers(None, 16, wl_set, cfg["n_cells"], 25)
    assert len(centres) == gold_c1["n_centres"]
    assert hashlib.sha256(np.asarray(centres, dtype=np.uint64).tobytes()).hexdigest() == gold_c1["centres_sha256"]
    bg.cluster(None, wl_set, cfg["n_cells"], 16, 25)
    assign = bg.assign_by_cluster(16)
    h = hashlib.sha256()
    for k in sorted(assign):
        h.update(("%s\t%s\n" % (k, assign[k])).encode())
    assert len(assign) == gold_c1["n_assigned"] and h.hexdigest() == gold_c1["assignments_sha256"]


def test_kmer_indexer_golden(gold_kmer):
    for c in gold_kmer:
        if len(c["query"]) != 16 or any(len(s) != 16 for s in c["known"]):
            continue
        got = KmerIndexer(c["known"], c["k"]).get_occurrences(c["query"], **c["kw"])
        assert [(k, v[1], list(v[2])) for k, v in got.items()] == [(x[0], x[1], x[2]) for x in c["result"]]


# ------------------------------------------------------------------------------------------ oracle, seeded inputs
@pytest.mark.parametrize("t", [1, 2, 3])
def test_edges_vs_oracle_clustered(t, mode):
    s = clustered_set(40 + t, 300, 30000 if t < 3 else 6000, 0.06)
    a, b, d = ops.edges_build(s, t)
    ix = orc.Index(s)
    wa, wb, wd, _ = ix.edges(t)
    assert np.array_equal(edge_rows(a, b, d), np.stack([wa, wb, wd], 1).astype(np.int64))
    assert a.size > 1000


@pytest.mark.parametrize("t", [1, 2])
def test_edges_dense_neighbourhoods(t, mode):
    """Consecutive integers and low-complexity families: every sub-tile next to the diagonal is dense."""
    rng = np.random.default_rng(5)
    base = int(rng.integers(0, 1 << 31))
    s = np.unique(np.concatenate([np.arange(base, base + 3000, dtype=np.uint64),
                                  (np.arange(0, 2500, dtype=np.uint64) << np.uint64(20)) + np.uint64(0x55555),
                                  rng.integers(0, 1 << 32, 4000, dtype=np.uint64)]).astype(np.uint32))
    a, b, d = ops.edges_build(s, t)
    wa, wb, wd, _ = orc.Index(s).edges(t)
    assert np.array_equal(edge_rows(a, b, d), np.stack([wa, wb, wd], 1).astype(np.int64))


def _structured_set(rng, kind, n):
    """Small barcode sets with structure that stresses the interval tests, the candidate queues and the pass hand-over."""
    if kind == 0:      # uniform random
        v = rng.integers(0, 1 << 32, n, dtype=np.uint64)
    elif kind == 1:    # one dense run of consecutive integers (every tile next to the diagonal is full of candidates)
        v = np.arange(n, dtype=np.uint64) + np.uint64(int(rng.integers(0, (1 << 32) - n)))
    elif kind == 2:    # few cells, many errors: real clusters
        cells = rng.integers(0, 1 << 32, max(2, n // 40), dtype=np.uint64).astype(np.uint32)
        v, _ = synth.simulate_reads(cells, n, 0.10, rng, star_frac=0.0)
        v = v.astype(np.uint64)
    elif kind == 3:    # shared high half / shared low half / shared middle: one block constant, the rest random
        which = int(rng.integers(0, 3))
        mask = [np.uint64(0xFFFF0000), np.uint64(0x0000FFFF), np.uint64(0x00FFFF00)][which]
        v = (rng.integers(0, 1 << 32, n, dtype=np.uint64) & ~mask) | (np.uint64(int(rng.integers(0, 1 << 32))) & mask)
    elif kind == 4:    # low complexity: periodic words with a few edits
        out = []
        for _ in range(n):
            unit = int(rng.integers(0, 1 << (2 * int(rng.integers(1, 4)))))
            ul = int(rng.integers(1, 4))
            w = 0
            for i in range(16):
                w |= ((unit >> (2 * (i % ul))) & 3) << (2 * i)
            for _e in range(int(rng.integers(0, 3))):
                w ^= int(rng.integers(1, 4)) << (2 * int(rng.integers(0, 16)))
            out.append(w)
        v = np.asarray(out, dtype=np.uint64)
    else:              # values at the ends of the range and around field boundaries of the rotated keys
        base = np.asarray([0, 1, 2, 3, 0xFFFFFFFF, 0xFFFFFFFE, 0x3FFFFFFF, 0x40000000, 0x7FFFFFFF, 0x80000000, 0xBFFFFFFF, 0xC0000000,
                           0x000FFFFF, 0x00100000, 0x0000FFFF, 0x00010000, 0x003FFFFF, 0x00400000], dtype=np.uint64)
        v = np.concatenate([base, base ^ np.uint64(0x55555555), rng.integers(0, 1 << 32, n, dtype=np.uint64)])
    return np.unique(v.astype(np.uint32))


@pytest.mark.parametrize("t", [1, 2])
def test_edges_many_small_structured_sets(t, mode):
    """Every pair decided by brute force (oracle predicate on all pairs) on many small sets of each structure."""
    rng = np.random.default_rng(100 + t)
    total = 0
    for trial in range(36):
        kind = trial % 6
        n = int(rng.integers(2, 1500)) if trial % 5 else int(rng.integers(1500, 3500))
        s = _structured_set(rng, kind, n)
        a, b, d = ops.edges_build(s, t)
        wa, wb, wd = orc.edges_brute(s, t)
        assert np.array_equal(edge_rows(a, b, d), np.stack([wa, wb, wd], 1).astype(np.int64)), (trial, kind, s.size)
        total += a.size
    assert total > 10000


def test_edges_edge_cases(mode):
    for t in (1, 2, 3):
        for arr in ([], [7], [0, 0xFFFFFFFF], [0, 1, 2, 3], list(range(2047, 2047 + 5))):
            s = np.asarray(arr, np.uint32)
            a, b, d = ops.edges_build(s, t)
            wa, wb, wd = orc.edges_brute(s, t)
            assert np.array_equal(edge_rows(a, b, d), np.stack([wa, wb, wd], 1).astype(np.int64))
    with pytest.raises(badger_b200.BadgerB200Error):
        ops.edges_build(np.asarray([5, 5, 6], np.uint32), 1)         # not strictly increasing
    with pytest.raises(badger_b200.BadgerB200Error):
        ops.edges_build(np.asarray([9, 3], np.uint32), 1)
    a, _, _ = ops.edges_build(np.arange(100, dtype=np.uint32), 0)    # t = 0: no edges (barcode_graph.py:245)
    assert a.size == 0


def test_edge_buffer_regrow(monkeypatch, mode):
    """The library sizes its edge buffer from a guess and re-runs the (deterministic) kernel when it was too small."""
    s = clustered_set(55, 40, 60000, 0.05)
    want = edge_rows(*ops.edges_build(s, 2))
    assert want.shape[0] > (1 << 16) + 1024 + s.size          # more edges than the forced guess below
    badger_b200.lib().bdg_shutdown()                            # drop the grown workspaces
    monkeypatch.setenv("BDG_EDGE_CAP_PER_ROW", "1")
    badger_b200.init()
    got = edge_rows(*ops.edges_build(s, 2))
    assert np.array_equal(got, want)


def test_tile_list_regrow(monkeypatch):
    """Sparse mode sizes its tile list from a guess; when the scan finds more tiles the list grows and the scan repeats."""
    s = clustered_set(56, 60, 50000, 0.05)
    L = badger_b200.lib()
    badger_b200._lib.check(L.bdg_set_edge_mode(1))
    want = edge_rows(*ops.edges_build(s, 2))
    L.bdg_shutdown()                                            # drop the grown workspaces
    monkeypatch.setenv("BDG_TILE_LIST_CAP", "8")
    badger_b200.init()
    got = edge_rows(*ops.edges_build(s, 2))
    badger_b200._lib.check(L.bdg_set_edge_mode(-1))
    assert want.shape[0] > 10000 and np.array_equal(got, want)


def test_stale_edge_handle_is_refused():
    """A handle's edges live in the device workspaces until copied; a later build on the device invalidates it."""
    s = clustered_set(57, 20, 3000, 0.05)
    L = badger_b200.lib()
    h1, h2 = C.c_void_p(), C.c_void_p()
    badger_b200._lib.check(L.bdg_edges_build(s.ctypes.data, s.size, 1, C.byref(h1)))
    n1 = L.bdg_edges_count(h1)
    badger_b200._lib.check(L.bdg_edges_build(s.ctypes.data, s.size, 1, C.byref(h2)))
    a = np.empty(n1, np.uint32); b = np.empty(n1, np.uint32); d = np.empty(n1, np.uint8)
    assert n1 > 0 and L.bdg_edges_copy(h1, a.ctypes.data, b.ctypes.data, d.ctypes.data) == badger_b200._lib.BDG_ERR_ARG
    assert L.bdg_edges_copy(h2, a.ctypes.data, b.ctypes.data, d.ctypes.data) == 0
    L.bdg_edges_free(h1); L.bdg_edges_free(h2)


@pytest.mark.parametrize("nparts", [1, 2, 3, 8])
def test_parts_union_equals_full(nparts, mode):
    """ops.edges_build_part is the streaming form (bdg_edges_build_into): nparts = 1 checks it against the resident form."""
    s = clustered_set(77, 200, 20000, 0.06)
    fa, fb, fd = ops.edges_build(s, 2)
    rows = []
    total_pairs = 0
    for p in range(nparts):
        a, b, d = ops.edges_build_part(s, 2, p, nparts)
        own = set(s[part_rows(s.size, p, nparts)].tolist())
        if mode == "dense":
            assert all(x in own for x in a.tolist())                  # dense: a part emits the edges of its own rows
        rows.append(edge_rows(a, b, d))
        pp = badger_b200.lib().bdg_part_pairs(s.size, p, nparts)
        assert pp == part_pairs(s.size, p, nparts)
        total_pairs += pp
    assert total_pairs == s.size * (s.size - 1) // 2
    merged = np.concatenate(rows)
    merged = merged[np.lexsort((merged[:, 1], merged[:, 0]))]
    assert np.array_equal(merged, edge_rows(fa, fb, fd))


def test_dedup_first_seen_vs_oracle():
    """Row a-2 on the device: same distinct order (first sighting), counts and read map as the oracle's restatement of
    barcode_graph.py:192-204."""
    rng = np.random.default_rng(21)
    for R, pool in ((1, 1), (2, 1), (1000, 10), (5000, 5000), (300000, 20000), (1 << 20, 1 << 18)):
        src = rng.integers(0, 1 << 32, pool, dtype=np.uint64).astype(np.uint32)
        src[: min(4, pool)] = np.asarray([0, 0xFFFFFFFF, 1, 0x80000000], np.uint32)[: min(4, pool)]
        reads = src[rng.integers(0, pool, R)]
        d, c, m, sp = ops.dedup_first_seen(reads, want_map=True, want_sorted_pos=True)
        wd, wc = orc.dedup_count(reads)
        assert np.array_equal(d, wd) and np.array_equal(c, np.asarray(wc, np.int64))
        assert np.array_equal(d[m], reads)                      # the map sends every read to its own barcode
        srt = np.empty_like(d); srt[sp] = d
        assert np.array_equal(srt, np.sort(d))                  # sorted_pos = position in ascending order
    d, c = ops.dedup_first_seen(np.empty(0, np.uint32))
    assert d.size == 0 and c.size == 0


def test_cluster_levels_vs_reference_rounds():
    """Row f-3 on the device against the literal restatement of barcode_graph.py:283-301 (oracle.cluster): random graphs
    with many same-round conflicts, centres that are not nodes, and a clustered barcode set with its real edges."""
    rng = np.random.default_rng(33)
    cases = []
    for trial in range(25):
        n = int(rng.integers(5, 400))
        s = np.sort(rng.choice(1 << 24, n, replace=False).astype(np.uint32))
        m = int(rng.integers(0, 5 * n))
        x = rng.integers(0, n, m); y = rng.integers(0, n, m)
        pairs = sorted({(min(i, j), max(i, j)) for i, j in zip(x.tolist(), y.tolist()) if i != j})
        ea = s[[p[0] for p in pairs]] if pairs else np.empty(0, np.uint32)
        eb = s[[p[1] for p in pairs]] if pairs else np.empty(0, np.uint32)
        cen = s[rng.choice(n, int(rng.integers(1, max(2, n // 3))), replace=False)]
        if trial % 3 == 0:
            cen = np.concatenate([cen, np.asarray([(1 << 24) + 5, (1 << 24) + 9], np.uint32)])     # never observed
        cases.append((s, ea, eb, cen))
    big = clustered_set(91, 300, 30000, 0.06)
    ba, bb, _ = ops.edges_build(big, 2)
    cases.append((big, ba, bb, big[rng.choice(big.size, 250, replace=False)]))
    for s, ea, eb, cen in cases:
        ci, lv = ops.cluster_levels(s, ea, eb, cen, 2)
        adj = {}
        for u, v in zip(ea.tolist(), eb.tolist()):
            adj.setdefault(u, []).append(v); adj.setdefault(v, []).append(u)
        want = orc.cluster(adj, [int(c) for c in cen.tolist()])
        pos = {int(v): i for i, v in enumerate(s.tolist())}
        got = {}
        for i in np.nonzero(ci != -2)[0].tolist():
            got[int(s[i])] = (int(s[ci[i]]), int(lv[i])) if ci[i] >= 0 else (-1, -1)
        assert got == {k: tuple(v) for k, v in want.items() if k in pos}
        # the mask behind `len(graph.edges.keys())` (badger.py:131): non-centre nodes with at least one edge
        ci2, lv2, has = ops.cluster_levels(s, ea, eb, cen, 2, want_has_edge=True)
        assert np.array_equal(ci2, ci) and np.array_equal(lv2, lv)
        deg = np.zeros(s.size, bool)
        deg[np.searchsorted(s, ea)] = True; deg[np.searchsorted(s, eb)] = True
        assert np.array_equal(has, deg & (lv != 0))
    assert any((ci == -1).any() for ci, _ in [ops.cluster_levels(*c, 2) for c in cases[:10]])      # conflicts were exercised


def test_dedup_reads_and_assign_reads_vs_numpy():
    """Rows f-1 / f-2 with the per-read arrays resident on the device (bdg_dedup_reads + bdg_assign_reads) against the
    host-array operators and a numpy restatement: masks of every kind, the token life cycle, bad sizes."""
    rng = np.random.default_rng(17)
    none = np.uint64(1) << np.uint64(32)
    for R, pool, pv in ((1, 1, 1.0), (5, 3, 0.5), (1000, 40, 0.9), (200000, 30000, 0.97), (200000, 5, 0.0), (77777, 70000, 1.0), (300001, 1000, 0.3)):
        keys = rng.integers(0, 1 << 32, pool, dtype=np.uint64).astype(np.uint32)
        ranks = keys[rng.integers(0, pool, R)]
        for valid in (None, rng.random(R) < pv):
            rm = ops.dedup_reads(ranks, valid)
            v = np.ones(R, bool) if valid is None else valid
            assert rm.n_valid == int(v.sum()) and rm.rows == R
            if rm.n_valid == 0:
                out, n = ops.assign_reads(rm, np.empty(0, np.int32))
                assert (out == none).all() and n == 0
                continue
            d, c, rmap, spos = ops.dedup_first_seen(ranks[v], want_map=True, want_sorted_pos=True)       # kills the token ...
            with pytest.raises(badger_b200.BadgerB200Error):
                ops.assign_reads(rm, np.zeros(d.size, np.int32))
            rm = ops.dedup_reads(ranks, valid)                                                            # ... so take a new one
            assert np.array_equal(rm.distinct, d) and np.array_equal(rm.counts, c) and np.array_equal(rm.sorted_pos, spos)
            assert np.array_equal(rm.sorted_distinct, np.sort(d))
            N = d.size
            s = np.sort(d)
            ci = rng.integers(-2, N, N).astype(np.int32)
            out, n = ops.assign_reads(rm, ci)
            cd = np.where(ci[spos] >= 0, s[np.maximum(ci[spos], 0)].astype(np.uint64), none)
            want = np.full(R, none, np.uint64)
            want[v] = cd[rmap]
            assert np.array_equal(out, want) and n == int((want != none).sum())
            out2, _ = ops.assign_reads(rm, ci)                                                            # the token survives its use
            assert np.array_equal(out2, want)
            with pytest.raises(badger_b200.BadgerB200Error):
                ops.assign_reads(rm, ci[:-1] if N > 1 else np.zeros(2, np.int32))
    rm = ops.dedup_reads(np.empty(0, np.uint32))
    assert rm.rows == 0 and ops.assign_reads(rm, np.empty(0, np.int32))[0].size == 0


def test_packed_pipeline_on_all_devices_matches_one_device():
    """SURVEY.md 8e: rows dealt to the GPUs, per-GPU edge lists gathered on the first device for the clustering rounds
    (bdg_cluster_levels_from_edges on a multi-device handle).  Needs >= 2 GPUs (gpurun --gpus 2)."""
    from badger_b200 import pipeline
    n_dev = badger_b200.init()
    many_devs = None if n_dev >= 2 else [0, 0]      # one GPU: two device contexts on it (own streams, workspaces, host threads, "peer" copies)
    rng = synth.rng_for(123)
    wl = synth.make_whitelist(50000, rng)
    cells = synth.pick_cells(wl, 1500, rng)
    obs, valid = synth.simulate_reads(cells, 300000, 0.05, rng)
    wls = np.sort(wl)
    res = {}
    try:
        for devs in ([0], many_devs):
            assert badger_b200.init(devs) == (1 if devs == [0] else max(n_dev, 2))
            for t, mode in ((1, -1), (2, -1), (2, 2)):                      # t = 2 also with the join form forced (the set is below its default size)
                badger_b200._lib.check(badger_b200.lib().bdg_set_edge_mode(mode))
                out, info = pipeline.assign_packed(obs, valid, threshold=t, n_cells=1500, whitelist_sorted=wls, high_sens=(t == 2 and mode == 2))
                s = synth.sorted_unique(obs[valid])
                h = ops.edges_handle(s, t)
                e = ops.canonical(*h.copy())
                ci, lv, has = h.cluster_levels(cells, 2, want_has_edge=True)
                h.free()
                res[(devs == [0], t, mode)] = (out, info, e, ci, lv, has)
    finally:
        badger_b200._lib.check(badger_b200.lib().bdg_set_edge_mode(-1))
        badger_b200.init()
    for t, mode in ((1, -1), (2, -1), (2, 2)):
        one, many = res[(True, t, mode)], res[(False, t, mode)]
        assert np.array_equal(one[0], many[0]) and one[1] == many[1]
        for x, y in zip(one[2], many[2]):
            assert np.array_equal(x, y)
        assert np.array_equal(one[3], many[3]) and np.array_equal(one[4], many[4]) and np.array_equal(one[5], many[5])
        assert one[1]["edges"] > 1000
    for x, y in zip(res[(True, 2, -1)][2], res[(True, 2, 2)][2]):          # and the two t = 2 routes agree
        assert np.array_equal(x, y)


def test_resident_stages_vs_host_arrays():
    """The stages that keep their per-barcode arrays on the device (centre head, clustering result, 5-byte per-read result,
    whitelist packing) against the operators that return host arrays and numpy restatements of barcode_graph.py:252-258."""
    from badger_b200 import pipeline
    rng = synth.rng_for(321)
    wl = synth.make_whitelist(40000, rng)
    cells = synth.pick_cells(wl, 1200, rng)
    obs, valid = synth.simulate_reads(cells, 250000, 0.05, rng)
    wls = np.sort(wl)
    # whitelist records -> sorted distinct packed barcodes on the device
    recs = np.frombuffer(b"".join(synth.unrank_many(wl).tolist()) + b"ACGTNNNNACGTACGT" + synth.unrank_many(wl[:5]).tobytes(), np.uint8).reshape(-1, 16)
    assert np.array_equal(ops.pack16_sorted(recs), wls)
    assert ops.pack16_sorted(np.empty((0, 16), np.uint8)).size == 0
    for n_cells in (1200, 50, 400000):
        rm = ops.dedup_reads(obs, valid)
        d, c = rm.distinct, rm.counts
        first = c[:n_cells]
        cutoff = max((int(first.sum()) / first.size) / 5.0, 5)
        above = np.nonzero(c > cutoff)[0]
        above = above[np.argsort(-c[above], kind="stable")]
        for w in (None, wls):
            cut, top, cnt, hits = ops.centres_above(rm, n_cells, w)
            assert cut == cutoff and np.array_equal(top, d[above]) and np.array_equal(cnt, c[above])
            assert (hits is None) == (w is None)
            if w is not None:
                assert np.array_equal(hits, np.isin(d[above], wls))
            from badger_b200.barcode_graph import rest_by_counts
            for need in (1, 7, 3000, 10 ** 9):                                # the stretch behind the head, count level by count level
                want = rest_by_counts(d, c, cutoff, min(need, d.size) - 1)[:need]
                assert np.array_equal(ops.centres_rest(rm, cut, need), want)
    # too few whitelisted barcodes above the cutoff: the walk tops the list up from below it (barcode_graph.py:273-276)
    few = np.sort(cells[:300])
    got = pipeline.select_centres(rm, 1200, 25, few, None)
    g = badger_b200.BarcodeGraph.from_arrays(2, rm.distinct, rm.counts, with_dict=False)
    tok = object()
    g._wl_cache = (tok, few)
    assert got == g.get_cluster_centers(None, 16, tok, 1200, 25) and len(got) >= 900
    with pytest.raises(badger_b200.BadgerB200Error):
        ops.centres_above(rm, 10, wls[::-1].copy())                          # whitelist not sorted
    for t in (1, 2):
        want, info = pipeline.assign_packed(obs, valid, threshold=t, n_cells=1200, whitelist_sorted=wls)
        (c32, has), info2 = pipeline.assign_packed(obs, valid, threshold=t, n_cells=1200, whitelist_sorted=wls, form="u32")
        assert info == info2 and np.array_equal(has.astype(bool), want != pipeline.NONE)
        assert np.array_equal(c32[has != 0].astype(np.uint64), want[want != pipeline.NONE])
        # the same through the host-array operators: edges copied out, clustering rounds from host arrays, 8-byte gather
        rm = ops.dedup_reads(obs, valid)
        s = rm.sorted_distinct
        a, b, _ = ops.edges_build(s, t)
        centres = np.asarray(list(dict.fromkeys(pipeline.select_centres(rm, 1200, 25, wls, None))), np.uint32)
        ci, lv, has_edge = ops.cluster_levels(s, a, b, centres, 2, want_has_edge=True)
        out, n = ops.assign_reads(rm, ci)
        assert np.array_equal(out, want) and n == info["assigned_reads"]
        assert info["disconnected"] == s.size - (int(has_edge.sum()) + centres.size) and info["edges"] == a.size
        with pytest.raises(badger_b200.BadgerB200Error):
            ops.assign_reads32(rm, None)                                     # no clustering result of this dedup is resident


def test_member_vs_oracle():
    rng = np.random.default_rng(8)
    for W in (0, 1, 5, 1000, 1024, 1025, 300000):
        wl = np.unique(rng.integers(0, 1 << 32, W, dtype=np.uint64).astype(np.uint32))
        q = np.concatenate([rng.integers(0, 1 << 32, 5000, dtype=np.uint64).astype(np.uint32), wl[:2000],
                            np.asarray([0, 0xFFFFFFFF], np.uint32)])
        assert np.array_equal(ops.member_sorted(wl, q), orc.member(wl, q).astype(bool))
    assert ops.member_sorted(np.asarray([1, 2], np.uint32), np.empty(0, np.uint32)).size == 0


@pytest.mark.parametrize("max_d", [2, 1, 0, 4])
def test_nearest_vs_oracle(max_d):
    rng = np.random.default_rng(9)
    centres = rng.integers(0, 1 << 32, 700, dtype=np.uint64).astype(np.uint32)
    obs, _ = synth.simulate_reads(centres, 4000, 0.08, rng)
    q = np.concatenate([obs, centres[:50], rng.integers(0, 1 << 32, 500, dtype=np.uint64).astype(np.uint32)])
    tg = np.concatenate([centres, centres[:30] ^ np.uint32(1)])       # near-duplicates force ties on distance
    tg = tg[rng.permutation(tg.size)]
    am, dist = ops.nearest_bounded(q, tg, max_d)
    wam, wdist = orc.nearest(q, tg, max_d)
    assert np.array_equal(am, wam) and np.array_equal(dist, wdist)
    assert (am >= 0).sum() > 100
    e_am, e_d = ops.nearest_bounded(q[:10], np.empty(0, np.uint32), 2)
    assert (e_am == -1).all() and (e_d == 255).all()


@pytest.mark.parametrize("max_d", [2, 1, 0])
def test_nearest_large_sparse_path(max_d, monkeypatch):
    """Q x W large enough for the sorted / tiled form of the scorer (bdg_api.cu launch_nearest_sparse): same answers as the
    brute-force kernel and as the oracle, including ties on distance (first index in caller order wins) and duplicates."""
    rng = np.random.default_rng(19 + max_d)
    centres = rng.integers(0, 1 << 32, 6000, dtype=np.uint64).astype(np.uint32)
    obs, _ = synth.simulate_reads(centres, 70000, 0.07, rng)
    q = np.concatenate([obs, centres[:500], rng.integers(0, 1 << 32, 3000, dtype=np.uint64).astype(np.uint32),
                        np.asarray([0, 0xFFFFFFFF, 0x55555555], np.uint32)])
    tg = np.concatenate([centres, centres[:200] ^ np.uint32(1), centres[:100], np.asarray([0, 0xFFFFFFFF], np.uint32)])
    tg = tg[rng.permutation(tg.size)]
    assert q.size * tg.size >= 1 << 24
    am, dist = ops.nearest_bounded(q, tg, max_d)
    monkeypatch.setenv("BDG_NEAREST_DENSE", "1")
    am2, dist2 = ops.nearest_bounded(q, tg, max_d)
    assert np.array_equal(am, am2) and np.array_equal(dist, dist2)
    sel = rng.choice(q.size, 6000, replace=False)
    wam, wdist = orc.nearest(q[sel], tg, max_d)
    assert np.array_equal(am[sel], wam) and np.array_equal(dist[sel], wdist)
    assert (am >= 0).sum() > 1000


@pytest.fixture(params=["postings", "scan"])
def kmer_form(request, monkeypatch):
    """Both forms of a-5: the 6-mer posting lists (default from 4096 strings on) and the scan of every string."""
    monkeypatch.setenv("BDG_KMER_POST_MIN_W", "0" if request.param == "postings" else str(1 << 40))
    return request.param


def test_kmer_score_vs_oracle(kmer_form):
    rng = np.random.default_rng(10)
    wl = rng.integers(0, 1 << 32, 3000, dtype=np.uint64).astype(np.uint32)
    wl[:20] = np.asarray([0, 0x55555555, 0xAAAAAAAA, 0xFFFFFFFF, 0x11111111] * 4, np.uint32)   # low complexity
    q = np.concatenate([wl[:40], rng.integers(0, 1 << 32, 300, dtype=np.uint64).astype(np.uint32)])
    for mk in (1, 4, 5):
        hq, hw, cnt, mult = ops.kmer_score(q, wl, min_kmers=mk)
        wc, wm = orc.kmer_score(q, wl)
        wq, ww = np.nonzero(wc >= mk)
        o = np.lexsort((hw, hq))
        assert np.array_equal(hq[o], wq) and np.array_equal(hw[o], ww)
        assert np.array_equal(cnt[o], wc[wq, ww]) and np.array_equal(mult[o], wm[wq, ww])
    _, hw, _, _ = ops.kmer_score(q[:5], wl, min_kmers=1, cap=3)       # capacity retry path
    assert hw.size >= 5


def test_kmer_postings_large_string_set():
    """The posting lists at a whitelist-like size: 300 k strings, queries one substitution / one shift away from entries, and the
    low-complexity words whose 6-mers repeat inside the word (listed once per string, walked once per query)."""
    rng = np.random.default_rng(13)
    wl = np.unique(rng.integers(0, 1 << 32, 300000, dtype=np.uint64).astype(np.uint32))
    wl[:6] = np.asarray([0, 0x55555555, 0xAAAAAAAA, 0xFFFFFFFF, 0x11111111, 0x1B1B1B1B], np.uint32)
    src = wl[rng.integers(0, wl.size, 40)]
    q = np.concatenate([wl[:8], src ^ (np.uint32(2) << (2 * rng.integers(0, 16, 40)).astype(np.uint32)), src[:20] << np.uint32(2),
                        src[20:] >> np.uint32(2)])
    ix = ops.KmerIndex(wl)
    for mk in (1, 4):
        hq, hw, cnt, mult = ix.query(q, min_kmers=mk)
        wc, wm = orc.kmer_score(q, wl)
        wq, ww = np.nonzero(wc >= mk)
        o = np.lexsort((hw, hq))
        assert np.array_equal(hq[o], wq) and np.array_equal(hw[o], ww)
        assert np.array_equal(cnt[o], wc[wq, ww]) and np.array_equal(mult[o], wm[wq, ww])
    ix.free()


def test_resident_kmer_index_many_queries(kmer_form):
    """KmerIndexer / QGramIndex keep their strings on the device (ops.KmerIndex): repeated queries, growth after append."""
    rng = np.random.default_rng(12)
    wl = rng.integers(0, 1 << 32, 5000, dtype=np.uint64).astype(np.uint32)
    ix = ops.KmerIndex(wl)
    for _ in range(5):
        q = wl[rng.integers(0, wl.size, 7)] ^ np.uint32(1 << int(rng.integers(0, 32)))
        hq, hw, cnt, mult = ix.query(q, min_kmers=3)
        wc, wm = orc.kmer_score(q, wl)
        wq, ww = np.nonzero(wc >= 3)
        o = np.lexsort((hw, hq))
        assert np.array_equal(hq[o], wq) and np.array_equal(hw[o], ww) and np.array_equal(cnt[o], wc[wq, ww])
    ix.free()
    known = [orc.unrank(int(x)) for x in wl[:300].tolist()]
    ki = KmerIndexer(known, 6)
    before = ki.get_occurrences(known[5], min_kmers=2)
    assert known[5] in before
    extra = orc.unrank(int(wl[4000]))
    ki.append(extra)
    after = ki.get_occurrences(extra, min_kmers=2)
    assert extra in after and after[extra][1] == 121 or after[extra][1] >= 11       # S(x,x) >= 11


# ------------------------------------------------------------------------------------------ full size: properties
def test_c2_full_size_properties(mode):
    """BASELINE config 2 at full size (1 M reads, t=1): sampled rows against the oracle's index walk, plus
    structural properties that do not depend on the size."""
    wl, cells, obs, valid, cfg = synth.make_dataset("C2")
    s = np.unique(obs[valid])
    a, b, d = ops.edges_build(s, cfg["threshold"])
    assert (a < b).all() and ((d >= 1) & (d <= cfg["threshold"])).all()
    key = (a.astype(np.uint64) << np.uint64(32)) | b.astype(np.uint64)
    assert np.unique(key).size == key.size                                # no duplicate edges
    assert np.isin(a, s).all() and np.isin(b, s).all()
    rng = np.random.default_rng(2)
    rows = np.sort(rng.choice(s.size, 2000, replace=False)).astype(np.uint32)
    wa, wb, wd, _ = orc.Index(s).edges(cfg["threshold"], rows=rows)
    sel = np.isin(a, s[rows])
    assert np.array_equal(edge_rows(a[sel], b[sel], d[sel]), np.stack([wa, wb, wd], 1).astype(np.int64))
    # idempotence / determinism: a second run gives the same set
    a2, b2, d2 = ops.edges_build(s, cfg["threshold"])
    assert np.array_equal(edge_rows(a, b, d), edge_rows(a2, b2, d2))
    # whitelist hits at full size: every cell barcode present in the data is found, random words are not
    hit = ops.member_sorted(np.sort(wl), s)
    assert np.array_equal(hit, orc.member(np.sort(wl), s).astype(bool))


def test_t2_large_sampled_rows(mode):
    """t=2 at N ~ 4e5 (the shape of configs 4/5, scaled): sampled rows against the oracle."""
    rng = synth.rng_for(31)
    wl = synth.make_whitelist(50000, rng)
    cells = synth.pick_cells(wl, 8000, rng)
    obs, valid = synth.simulate_reads(cells, 900000, 0.05, rng)
    s = np.unique(obs[valid])
    a, b, d = ops.edges_build(s, 2)
    rows = np.sort(rng.choice(s.size, 1500, replace=False)).astype(np.uint32)
    assert_sampled_rows(s, a, b, d, rows, 2)
    assert (d == 2).sum() > 1000 and (d == 1).sum() > 1000


def assert_sampled_rows(s, a, b, d, rows, t):
    """The edges that touch the sampled rows - as the smaller OR the larger barcode - against the oracle's index walk
    (index.py:77-93 + barcode_graph.py:233-249) over the full array: SURVEY.md 0.6(ii)."""
    wa, wb, wd = orc.edges_touching(orc.Index(s), t, rows)
    picked = np.zeros(s.size, bool)
    picked[rows] = True
    sel = picked[np.searchsorted(s, a)] | picked[np.searchsorted(s, b)]
    assert np.array_equal(edge_rows(a[sel], b[sel], d[sel]), np.stack([wa, wb, wd], 1).astype(np.int64))
    assert wa.size > rows.size


@pytest.mark.parametrize("name", ["C4", "C5r1"])
def test_full_size_t2_sampled_rows(name):
    """BASELINE config 4 (2e7 reads, 4.6e6 distinct) and config 5 at ONT's error rate (1e8 reads, 1.6e7 distinct; the named
    5e7-distinct shape holds 2e9 edges = 18 GB of host arrays and is run by tools/run_configs.py instead), t = 2, at FULL size on
    the default route (join form): 1 500 sampled rows as either end point against the oracle, plus size-independent properties."""
    import os
    workers = min(32, len(os.sched_getaffinity(0)))
    wl, cells, obs, valid, cfg = synth.make_dataset(name, workers=workers)
    s = synth.sorted_unique(obs[valid])
    del obs, valid
    a, b, d = ops.edges_build(s, cfg["threshold"])
    assert a.size > 20 * s.size
    assert (a < b).all() and ((d >= 1) & (d <= 2)).all()
    rows = np.sort(np.random.default_rng(12).choice(s.size, 1500, replace=False)).astype(np.uint32)
    assert_sampled_rows(s, a, b, d, rows, cfg["threshold"])
    # no edge twice: the (a, b) keys of a 1/64 slice of the key space are distinct
    part = (a & np.uint32(63)) == 7
    key = (a[part].astype(np.uint64) << np.uint64(32)) | b[part].astype(np.uint64)
    assert np.unique(key).size == key.size
