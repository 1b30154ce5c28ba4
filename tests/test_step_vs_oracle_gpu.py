"""The correction step after the edge list, on the GPU, against the CPU oracle at the sizes where kernels go wrong.

- The whole step (pipeline.assign_packed, device.assign_packed, distributed.assign_packed in a world of one, two device contexts)
  against the same step run through the oracle-backed stand-ins of tests/cpu_ops.py: element for element, with `info`.
- The clustering rounds (ops.cluster_levels, EdgeHandle.cluster_levels, cluster_resident + assign_reads32, the bdg_dev_cluster_*
  phases) against oracle.cluster, the literal restatement of barcode_graph.py:283-301, on graphs that span every high half of
  the node table, hold a high half with tens of thousands of nodes, and put 2 ... 64 centres on one node in the same round.
- pack16 / pack16_sorted at the letter level: every byte value at every position, around the kernel's 1024-record blocks.
- Guard bands around every caller-owned output of the bdg_dev_* entry points: nothing is written outside the caller's buffer.

The tests without the gpu mark pin the references themselves (the numpy pack16, the graph generators) on the CPU."""
import ctypes as C

import numpy as np
import pytest
import torch

import badger_b200
import cpu_ops
from badger_b200 import device as bd
from badger_b200 import ops, pipeline, synth
from gpu_helpers import claimed, cuda, host
from oracle import oracle as orc

gpu = pytest.mark.gpu


def contexts():
    """Device lists for one context and for two: every device when the box has two or more, else two contexts on device 0."""
    n = badger_b200.init()
    return [[0], None if n >= 2 else [0, 0]]


# ================================================================================================= 1. the whole step vs the oracle
# N (distinct valid barcodes) sits above the default join thresholds (150 000 at t = 2, 90 000 at t = 3), so the default routes
# run.  The oracle's edge list of a dataset is built once and shared by all its variants.
DATASETS = {
    "C2_t1": dict(config="C2", reads=1_000_000, t=1),             # the round-1 headline config, sparse form; N ~ 4.9e5
    "C4_t2": dict(config="C4", reads=1_000_000, t=2),             # join form, realistic clouds; N ~ 4.6e5
    "C5_t2": dict(config="C5", reads=600_000, t=2),               # perr 0.128: many same-round conflicts, many lone nodes; N ~ 5e5
    "C4_t3": dict(config="C4", reads=400_000, t=3),               # t = 3 join; N ~ 2.2e5
}
JOIN_MIN_N = {1: 0, 2: 150_000, 3: 90_000}
VARIANTS = ["whitelist", "none", "true_barcodes", "high_sens"]
STEP_CASES = [(d, v) for d in DATASETS for v in VARIANTS if v != "high_sens" or DATASETS[d]["t"] <= 2 and d != "C5_t2"]


class OracleEdges:
    """The oracle's edge list of one barcode set and its adjacency, standing in for ops.EdgeHandle; the clustering rounds run
    through oracle.cluster on every call.  `last` keeps the (centre_idx, level) of the last clustering for the vacuity checks."""

    def __init__(self, s, t):
        self.s = s
        a, b, _, _ = orc.Index(s).edges(t)
        self.count, self.n_nodes = int(a.size), int(s.size)
        ends = np.concatenate([a, b])
        other = np.concatenate([b, a])
        order = np.argsort(ends, kind="stable")
        keys, starts = np.unique(ends[order], return_index=True)
        nbrs = np.split(other[order], starts[1:])
        self.adj = dict(zip(keys.tolist(), (x.tolist() for x in nbrs)))
        self.deg = np.zeros(s.size, bool)
        self.deg[np.searchsorted(s, keys)] = True
        self.last = None

    def cluster_levels(self, centres, rounds=2, want_has_edge=False):
        assert rounds == 2
        res = orc.cluster(self.adj, [int(c) for c in np.asarray(centres).tolist()])
        nodes = np.fromiter(res.keys(), np.int64, len(res))
        cen = np.asarray([v[0] for v in res.values()], np.int64)
        lev = np.asarray([v[1] for v in res.values()], np.int64)
        p = np.searchsorted(self.s, nodes)
        node = (p < self.s.size) & (self.s[np.minimum(p, self.s.size - 1)] == nodes)     # a centre never observed has no node
        p, cen, lev = p[node], cen[node], lev[node]
        ci = np.full(self.s.size, -2, np.int32)
        lv = np.full(self.s.size, 255, np.uint8)
        ev = cen == -1
        ci[p[ev]] = -1
        ci[p[~ev]] = np.searchsorted(self.s, cen[~ev])
        lv[p[~ev]] = lev[~ev]
        self.last = (ci.copy(), lv.copy())
        return (ci, lv, self.deg & (lv != 0)) if want_has_edge else (ci, lv)

    def cluster_resident(self, centres, rounds=2):
        ci, lv, has = self.cluster_levels(centres, rounds, True)
        cpu_ops._RESIDENT["ci"] = ci
        return int(has.sum())

    def free(self):
        pass


_DATA = {}


def step_data(name):
    """(whitelist ascending, cells, reads, valid, N, OracleEdges) of a dataset, made once per session."""
    if name not in _DATA:
        d = DATASETS[name]
        wl, cells, obs, valid, _ = synth.make_dataset(d["config"], reads=d["reads"])
        s = synth.sorted_unique(obs[valid])
        assert s.size > JOIN_MIN_N[d["t"]], "N must sit above the default join threshold"
        _DATA[name] = dict(wl=np.sort(wl), cells=cells, obs=obs, valid=valid, s=s, edges=OracleEdges(s, d["t"]), oracle={})
    return _DATA[name]


def step_kwargs(name, variant):
    D, d = step_data(name), DATASETS[name]
    kw = dict(threshold=d["t"], n_cells=synth.CONFIGS[d["config"]]["n_cells"], whitelist_sorted=D["wl"])
    if variant == "none":
        kw["whitelist_sorted"] = None
    elif variant == "true_barcodes":
        kw["true_barcodes"] = D["cells"].tolist()
    elif variant == "high_sens":
        kw["high_sens"] = True
    return kw


def oracle_step(name, variant, monkeypatch):
    """pipeline.assign_packed(form="u32") with every operator replaced by its oracle stand-in: ((centre, has), info), and the
    (centre_idx, level) of its clustering.  Memoised per (dataset, variant)."""
    D = step_data(name)
    if variant not in D["oracle"]:
        cpu_ops.install(monkeypatch)
        edges = D["edges"]

        def resident(rm, t):
            assert np.array_equal(rm.sorted_distinct, edges.s)
            return edges

        monkeypatch.setattr(ops, "edges_handle_resident", resident)
        try:
            out, info = pipeline.assign_packed(D["obs"], D["valid"], form="u32", **step_kwargs(name, variant))
        finally:
            monkeypatch.undo()
        D["oracle"][variant] = (out, info, edges.last)
    return D["oracle"][variant]


def as_u64(c32, has):
    out = c32.astype(np.uint64)
    out[has == 0] = pipeline.NONE
    return out


def assert_same(got, want):
    (c32, has), info = got
    (wc, wh), winfo = want
    assert np.array_equal(np.asarray(has).astype(bool), wh.astype(bool))
    assert np.array_equal(np.asarray(c32), wc)                    # 0 where there is no centre, on both sides
    assert info == winfo


def assert_not_vacuous(name, variant, monkeypatch):
    (_, has), info, (ci, lv) = oracle_step(name, variant, monkeypatch)
    counts = dict(evicted=int((ci == -1).sum()), level2=int((lv == 2).sum()), disconnected=info["disconnected"],
                  assigned=info["assigned_reads"], distinct=info["distinct"], edges=info["edges"])
    if variant == "high_sens":
        counts["high_sens_moved"] = info["assigned_reads"] - oracle_step(name, "whitelist", monkeypatch)[1]["assigned_reads"]
        assert counts["high_sens_moved"] > 0
    print("step counts %s/%s: %s" % (name, variant, counts))
    assert counts["evicted"] > 0 and counts["level2"] > 0 and counts["disconnected"] > 0
    assert info["valid_reads"] > info["assigned_reads"] > 0


@gpu
@pytest.mark.parametrize("name,variant", STEP_CASES)
def test_step_matches_oracle(name, variant, claimed, monkeypatch):
    D = step_data(name)
    want = oracle_step(name, variant, monkeypatch)
    assert_not_vacuous(name, variant, monkeypatch)
    kw = step_kwargs(name, variant)
    got = pipeline.assign_packed(D["obs"], D["valid"], form="u32", **kw)
    assert_same(got, want[:2])
    out64, info64 = pipeline.assign_packed(D["obs"], D["valid"], **kw)
    assert out64.dtype == np.uint64 and np.array_equal(out64, as_u64(*want[0])) and info64 == want[1]


@gpu
def test_step_on_tensors_two_contexts_and_world_of_one_match_oracle(claimed, monkeypatch):
    """On one t = 2 set: device.assign_packed on tensors, pipeline.assign_packed on two device contexts, and
    distributed.assign_packed without a process group (bdg_dev_dedup_merge and the bdg_dev_cluster_* phases), each against
    the oracle, for the whitelist and the high_sens variant."""
    from badger_b200 import distributed as bdist
    name = "C4_t2"
    D = step_data(name)
    for variant in ("whitelist", "high_sens"):
        want = oracle_step(name, variant, monkeypatch)[:2]
        kw = step_kwargs(name, variant)
        tkw = dict(kw, whitelist_sorted=cuda(kw["whitelist_sorted"]))
        for devs in contexts():
            badger_b200.init(devs)
            assert_same(pipeline.assign_packed(D["obs"], D["valid"], form="u32", **kw), want)
            (c, h), info = bd.assign_packed(cuda(D["obs"]), cuda(D["valid"], torch.bool), **tkw)
            assert_same(((host(c), host(h)), info), want)
        badger_b200.init([0])
        (c, h), info = bdist.assign_packed(cuda(D["obs"], torch.uint32), cuda(D["valid"], torch.bool), **tkw)
        assert_same(((host(c), host(h)), info), want)


# ================================================================================================= 2. the clustering rounds
def reference_rounds(s, ea, eb, cen):
    """oracle.cluster turned into node arrays: (centre_idx, level, has_edge) as ops.cluster_levels(..., want_has_edge=True)."""
    adj = {}
    for u, v in zip(np.asarray(ea).tolist(), np.asarray(eb).tolist()):
        adj.setdefault(u, []).append(v); adj.setdefault(v, []).append(u)
    res = orc.cluster(adj, [int(c) for c in np.asarray(cen).tolist()])
    pos = {int(v): i for i, v in enumerate(s.tolist())}
    ci = np.full(s.size, -2, np.int32); lv = np.full(s.size, 255, np.uint8)
    for node, (c, level) in res.items():
        if node in pos:
            ci[pos[node]] = -1 if c == -1 else pos[c]
            lv[pos[node]] = 255 if c == -1 else level
    has = np.zeros(s.size, bool)
    if len(ea):
        has[np.searchsorted(s, ea)] = True; has[np.searchsorted(s, eb)] = True
    return ci, lv, has & (lv != 0), adj, res


def claim_sizes(adj, res):
    """For every node oracle.cluster evicted: (round, number of distinct centres that claimed it in that round), measured on
    the result: round 1 if two or more centres are its neighbours, else round 2 through its level-1 neighbours."""
    out = []
    for node, (c, _) in res.items():
        if c != -1:
            continue
        nb = adj.get(node, ())
        r1 = {res[x][0] for x in nb if x in res and res[x][1] == 0}
        if len(r1) >= 2:
            out.append((1, len(r1)))
        else:
            out.append((2, len({res[x][0] for x in nb if x in res and res[x][1] == 1})))
    return out


def node_values(rng, kind):
    """Node barcodes (ascending, distinct).  kind "full": every one of the 65 536 high halves holds nodes; "gaps": long
    stretches of empty high halves.  Both hold 0 and 0xFFFFFFFF and one high half with 40 000 nodes."""
    hi = np.arange(1 << 16, dtype=np.uint32)
    if kind == "gaps":
        keep = np.ones(hi.size, bool)
        for lo, n in ((1, 9000), (20000, 3000), (30001, 1), (40000, 20000), (65000, 535)):
            keep[lo:lo + n] = False
        hi = hi[keep]
    one = (hi << np.uint32(16)) | rng.integers(0, 1 << 16, hi.size, dtype=np.uint32)
    dense_hi = 0x1234 if kind == "full" else 0xFFFF
    dense = (np.uint32(dense_hi) << np.uint32(16)) | rng.choice(1 << 16, 40000, replace=False).astype(np.uint32)
    return synth.sorted_unique(np.concatenate([one, dense, np.asarray([0, 0xFFFFFFFF, 1, 0xFFFFFFFE], np.uint32)]))


def adversarial_graph(seed, kind):
    """(nodes, ea, eb, centres) of a generated graph (node_values) with:
    - hubs claimed in round 1 by k = 2 ... 64 centres at once, and nodes claimed in round 2 by k level-1 nodes of k centres;
    - a node joined in round 1 that a round-2 path from another centre also reaches;
    - centre-centre edges, centres that are no node, edges listed twice and in both orientations;
    - random edges inside the dense high half and across the whole range, 0 and 0xFFFFFFFF as centres and edge ends."""
    rng = np.random.default_rng(seed)
    s = node_values(rng, kind)
    n = s.size
    perm = rng.permutation(np.arange(2, n - 2))                  # node positions; 0 / 1 and n-2 / n-1 are placed by hand
    it = iter(perm[:12000].tolist())                             # the hand-made shapes take their nodes from here ...
    rest = np.sort(perm[12000:])                                 # ... and the random edges and centres from here only
    ea, eb, cen = [], [], []

    def edge(u, v):
        ea.append(u); eb.append(v)

    for k in list(range(2, 65)) + [64, 33, 17, 5, 2]:
        hub = next(it)                                           # round 1: k centres claim the hub
        cs = [next(it) for _ in range(k)]
        cen += cs
        for c in cs:
            edge(c, hub)
        hub2 = next(it)                                          # round 2: k centres, each over its own level-1 node
        for _ in range(k):
            c, mid = next(it), next(it)
            cen.append(c); edge(c, mid); edge(mid, hub2)
    # a node joined in round 1 (by c1) that c2's level-1 node also reaches in round 2: it stays c1's
    for _ in range(20):
        c1, c2, x, m = next(it), next(it), next(it), next(it)
        cen += [c1, c2]; edge(c1, x); edge(c2, m); edge(m, x)
    # centre-centre edges
    for _ in range(20):
        c1, c2 = next(it), next(it)
        cen += [c1, c2]; edge(c1, c2)
    # the extremes: 0 is a centre with neighbours, 0xFFFFFFFF a node claimed by two centres (and 0xFFFFFFFE reached from it)
    cen.append(0); edge(0, 1); edge(next(it), 0)
    c1, c2 = next(it), next(it)
    cen += [c1, c2]; edge(c1, n - 1); edge(n - 1, c2); edge(n - 1, n - 2)
    # random edges inside the dense high half (neighbours within 40 places) and over the whole range
    hi = (s[rest] >> np.uint32(16)).astype(np.int64)
    dense = rest[hi == np.bincount(hi).argmax()]
    x = rng.integers(0, dense.size, 60000)
    y = np.minimum(x + rng.integers(1, 40, x.size), dense.size - 1)
    ea += dense[x].tolist(); eb += dense[y].tolist()
    ea += rng.choice(rest, 60000).tolist(); eb += rng.choice(rest, 60000).tolist()
    cen += rng.choice(dense, 300, replace=False).tolist() + rng.choice(rest, 3000, replace=False).tolist()
    ea, eb = np.asarray(ea, np.int64), np.asarray(eb, np.int64)
    keep = ea != eb
    ea, eb = ea[keep], eb[keep]
    dup = rng.choice(ea.size, 3000, replace=False)
    swap = rng.random(ea.size) < 0.5                              # both orientations
    ea, eb = np.where(swap, eb, ea), np.where(swap, ea, eb)
    ea = np.concatenate([ea, ea[dup[:1500]], eb[dup[1500:]]])     # listed twice: as it was, and reversed
    eb = np.concatenate([eb, eb[dup[:1500]], ea[dup[1500:]]])
    cen = s[np.asarray(list(dict.fromkeys(cen)), np.int64)]
    missing = np.setdiff1d(rng.integers(0, 1 << 32, 64, dtype=np.uint64).astype(np.uint32), s)[:20]
    cen = np.concatenate([cen, missing])                          # centres that were never observed
    rng.shuffle(cen)
    return s, s[ea], s[eb], cen


GRAPHS = [(11, "full"), (12, "gaps")]


@pytest.mark.parametrize("seed,kind", GRAPHS)
def test_graph_generators_make_what_they_claim(seed, kind):
    s, ea, eb, cen = adversarial_graph(seed, kind)
    hi = np.unique(s >> np.uint32(16))
    assert s.size > 1 << 16 and s[0] == 0 and s[-1] == 0xFFFFFFFF and np.all(np.diff(s.astype(np.int64)) > 0)
    assert np.bincount((s >> np.uint32(16)).astype(np.int64)).max() >= 40000               # one high half, full-length search
    if kind == "full":
        assert hi.size == 1 << 16
    else:
        gaps = np.diff(hi.astype(np.int64)) - 1
        assert gaps.max() >= 9000 and (gaps > 0).sum() >= 4 and hi[0] == 0 and hi[-1] == 0xFFFF
    assert {0, 0xFFFFFFFF} <= set(np.concatenate([ea, eb]).tolist()) and 0 in set(cen.tolist())
    assert (~np.isin(cen, s)).sum() >= 10                                                   # centres that are no node
    key = np.minimum(ea, eb).astype(np.uint64) << np.uint64(32) | np.maximum(ea, eb).astype(np.uint64)
    assert np.unique(key).size < key.size and (ea > eb).any() and (ea < eb).any()           # duplicates, both orientations
    cs = set(cen.tolist())
    assert sum(1 for u, v in zip(ea.tolist(), eb.tolist()) if u in cs and v in cs) >= 20   # centre-centre edges
    _, lv, _, adj, res = reference_rounds(s, ea, eb, cen)
    sizes = claim_sizes(adj, res)
    by_round = {r: {k for rr, k in sizes if rr == r} for r in (1, 2)}
    assert set(range(2, 65)) <= by_round[1] and set(range(2, 65)) <= by_round[2], by_round
    assert res[0xFFFFFFFF][0] == -1 and res[0] == (0, 0)
    assert (lv == 2).sum() > 1000 and (lv == 1).sum() > 1000


@gpu
@pytest.mark.parametrize("seed,kind", GRAPHS)
def test_cluster_levels_on_adversarial_graphs(seed, kind, claimed):
    """ops.cluster_levels (host arrays) and the bdg_dev_cluster_* phases (distributed.cluster_levels, a world of one) on the
    generated graphs, against oracle.cluster; an edge end that is not a node is refused by both."""
    from badger_b200 import distributed as bdist
    s, ea, eb, cen = adversarial_graph(seed, kind)
    want_ci, want_lv, want_has, _, _ = reference_rounds(s, ea, eb, cen)
    for devs in contexts():
        badger_b200.init(devs)
        ci, lv, has = ops.cluster_levels(s, ea, eb, cen, 2, want_has_edge=True)
        assert np.array_equal(ci, want_ci) and np.array_equal(lv, want_lv) and np.array_equal(has, want_has)
    badger_b200.init([0])
    dci, dlv = bdist.cluster_levels(cuda(s), cuda(ea), cuda(eb), cen)
    dci, dlv = host(dci).astype(np.int32), host(dlv)
    assert np.array_equal(dci, want_ci)
    assert np.array_equal(np.where(dlv == ops.LEVEL_HAS_EDGE, 255, dlv), want_lv)
    assert np.array_equal((dlv != 255) & (dlv != 0), want_has)
    # an end point that is not a node: values near both ends of the range, one beside a node, one in an empty high half (gaps)
    absent = np.setdiff1d(np.asarray([5, 0xFFFFFFFD, int(s[s.size // 2]) + 1, 0x00020000], np.uint32), s)
    for v in absent:
        bad_a = np.concatenate([ea, [v]]).astype(np.uint32)
        bad_b = np.concatenate([eb, [s[3]]]).astype(np.uint32)
        with pytest.raises(badger_b200.BadgerB200Error):
            ops.cluster_levels(s, bad_a, bad_b, cen, 2)
        with pytest.raises(badger_b200.BadgerB200Error):
            bdist.cluster_levels(cuda(s), cuda(bad_b), cuda(bad_a), cen)
    ci, lv = ops.cluster_levels(s, ea, eb, cen, 2)                                        # and the library still works
    assert np.array_equal(ci, want_ci)


def barcode_graph_nodes(rng):
    """A barcode set whose real edges (t = 1) span every high half and hold dense stretches and hubs: one barcode in each of
    the 65 536 high halves, 40 000 in one high half (single-letter neighbours among them everywhere), 0 and 0xFFFFFFFF with neighbours, and
    hubs with 2 ... 48 single-substitution neighbours, which the test makes centres."""
    hi = np.arange(1 << 16, dtype=np.uint32)
    one = (hi << np.uint32(16)) | rng.integers(0, 1 << 16, hi.size, dtype=np.uint32)
    dense = np.uint32(0xB00B << 16) | rng.choice(1 << 16, 40000, replace=False).astype(np.uint32)
    hubs = rng.integers(0, 1 << 32, 48, dtype=np.uint64).astype(np.uint32)
    subs, hub_centres = [], []
    for k, h in zip(range(2, 49), hubs.tolist()):
        opts = [(h & ~(3 << (2 * p))) | (((h >> (2 * p)) + d) & 3) << (2 * p) for p in range(16) for d in (1, 2, 3)]
        pick = [opts[i] for i in rng.choice(len(opts), k, replace=False)]
        subs += pick; hub_centres.append(pick)
    ext = np.asarray([0, 1, 4, 0xFFFFFFFF, 0xFFFFFFFE, 0x3FFFFFFF], np.uint32)
    s = synth.sorted_unique(np.concatenate([one, dense, hubs, np.asarray(subs, np.uint32), ext]))
    return s, np.asarray(sum(hub_centres, []), np.uint32)


@gpu
def test_edge_handle_rounds_and_resident_gather_vs_oracle(claimed):
    """EdgeHandle.cluster_levels, and cluster_resident followed by assign_reads32 (8- and 5-byte forms, on host arrays and on
    tensors), on a barcode set built for the node table's edges (barcode_graph_nodes), on one context and on two."""
    rng = np.random.default_rng(21)
    s, hub_centres = barcode_graph_nodes(rng)
    a, b, _, _ = orc.Index(s).edges(1)
    cen = np.concatenate([hub_centres, [0, 0xFFFFFFFF, 0x12345678], rng.choice(s, 6000, replace=False)]).astype(np.uint32)
    cen = np.asarray(list(dict.fromkeys(cen.tolist())), np.uint32)
    want_ci, want_lv, want_has, adj, res = reference_rounds(s, a, b, cen)
    assert (want_ci == -1).sum() > 100 and (want_lv == 2).sum() > 100
    assert max(k for _, k in claim_sizes(adj, res)) >= 40
    reads = np.concatenate([s, s[rng.integers(0, s.size, 2 * s.size)]])     # every node in a valid row, then repeats
    valid = np.concatenate([np.ones(s.size, bool), rng.random(2 * s.size) < 0.9])
    p = rng.permutation(reads.size)
    reads, valid = reads[p], valid[p]
    for devs in contexts():
        badger_b200.init(devs)
        h = ops.edges_handle(s, 1)
        assert h.count == a.size
        ci, lv, has = h.cluster_levels(cen, 2, want_has_edge=True)
        assert np.array_equal(ci, want_ci) and np.array_equal(lv, want_lv) and np.array_equal(has, want_has)
        rm = ops.dedup_reads(reads, valid)
        assert np.array_equal(rm.sorted_distinct, s)
        h = ops.edges_handle_resident(rm, 1)
        assert h.n_nodes == s.size and h.count == a.size
        assert h.cluster_resident(cen, 2) == int(want_has.sum())
        centre = np.where(want_ci >= 0, s[np.maximum(want_ci, 0)], 0).astype(np.uint32)
        node = np.searchsorted(s, reads)
        want_c = np.where(valid & (want_ci[node] >= 0), centre[node], 0).astype(np.uint32)
        want_h = (valid & (want_ci[node] >= 0)).astype(np.uint8)
        c32, h8, n = ops.assign_reads32(rm, None)
        assert np.array_equal(h8, want_h) and np.array_equal(c32, want_c) and n == int(want_h.sum())
        out, n = ops.assign_reads(rm, ci)
        assert np.array_equal(out, as_u64(want_c, want_h)) and n == int(want_h.sum())
        # the same read map through the tensor gather with a device centre_idx
        got_c = torch.empty(reads.size, dtype=torch.int32, device=bd._device())
        got_h = torch.empty(reads.size, dtype=torch.bool, device=bd._device())
        d_ci = torch.from_numpy(ci).to(bd._device())
        nn = C.c_size_t(0)
        badger_b200._lib.check(badger_b200.lib().bdg_dev_assign_reads32(rm.token, d_ci.data_ptr(), s.size, got_c.data_ptr(),
                                                                        got_h.data_ptr(), reads.size, C.byref(nn), bd._stream()))
        assert np.array_equal(host(got_h), want_h.astype(bool)) and np.array_equal(host(got_c), want_c) and nn.value == n


# ================================================================================================= 3. pack16 at the letter level
ACGT = np.frombuffer(b"ACGT", np.uint8)
PACK_SIZES = [1, 3, 255, 256, 257, 1023, 1024, 1025, 4097, (1 << 22) + 5]


def ref_pack16(recs):
    """common.rank over uint8[R, 16] records: valid iff every byte is one of b"ACGT"; rank = sum(code_i * 4**i)."""
    lut = np.full(256, 255, np.uint8)
    lut[ACGT] = np.arange(4, dtype=np.uint8)
    codes = lut[recs]
    valid = (codes != 255).all(1)
    r = np.zeros(recs.shape[0], np.uint32)
    for i in range(16):
        r |= (codes[:, i] & np.uint8(3)).astype(np.uint32) << np.uint32(2 * i)
    return r, valid


def every_byte_everywhere(rng):
    """4 096 records: an otherwise valid record with byte value v at position p, for every v in 0 ... 255 and p in 0 ... 15."""
    base = ACGT[rng.integers(0, 4, 16)]
    recs = np.tile(base, (4096, 1))
    v = np.arange(4096) % 256
    p = np.arange(4096) // 256
    recs[np.arange(4096), p] = v
    return recs


def random_records(rng, n):
    """Records over ACGT with, per byte, a 3 % chance of one of b"Nacgt\\n\\0" or a high byte (0x80 ... 0xFF; the high bit set on
    a letter, 0xC1 / 0xC3 / 0xC7 / 0xD4, too)."""
    bad = np.frombuffer(b"Nacgt\n\0\xc1\xc3\xc7\xd4\x80\xff\xe1", np.uint8)
    recs = ACGT[rng.integers(0, 4, (n, 16))]
    m = rng.random((n, 16)) < 0.03
    recs[m] = bad[rng.integers(0, bad.size, int(m.sum()))]
    return recs


@pytest.fixture(scope="module")
def pack_pool():
    rng = np.random.default_rng(1616)
    ex = every_byte_everywhere(rng)
    return np.ascontiguousarray(np.concatenate([ex, random_records(rng, PACK_SIZES[-1] + 4096)]))


def oracle_pack16(recs):
    """orc.rank record by record (a high byte reaches it as a non-ASCII character, which it refuses as it refuses any letter
    outside ACGT)."""
    out = np.zeros(recs.shape[0], np.uint32); ok = np.zeros(recs.shape[0], bool)
    for i, rec in enumerate(recs):
        try:
            out[i], ok[i] = orc.rank(rec.tobytes().decode("latin-1")), True
        except KeyError:
            pass
    return out, ok


def test_ref_pack16_agrees_with_the_oracle_rank():
    rng = np.random.default_rng(5)
    recs = np.concatenate([every_byte_everywhere(rng), random_records(rng, 3000)])
    r, ok = ref_pack16(recs)
    wr, wok = oracle_pack16(recs)
    assert np.array_equal(ok, wok) and np.array_equal(r[ok], wr[ok])
    assert ok[:4096].sum() == 16 * 4 and 0 < ok[4096:].sum() < 3000          # 4 valid letters at each of 16 positions
    ascii_rows = (recs < 0x80).all(1)
    cr, cok = cpu_ops.pack16(recs[ascii_rows])
    assert np.array_equal(cok, ok[ascii_rows]) and np.array_equal(cr[cok], r[ascii_rows][cok])
    assert int(ref_pack16(np.frombuffer(b"ACGTACGTACGTACGT", np.uint8).reshape(1, 16))[0][0]) == 3840206052


@gpu
@pytest.mark.parametrize("n", PACK_SIZES)
def test_pack16_every_byte_at_every_position(n, pack_pool, claimed):
    for start in sorted({0, 4096 - min(n, 4096) // 2, 4096}):           # the exhaustive records, their seam, the random ones
        recs = pack_pool[start:start + n]
        want_r, want_ok = ref_pack16(recs)
        r, ok = ops.pack16(recs)
        assert np.array_equal(ok, want_ok) and np.array_equal(r[ok], want_r[ok])
        assert np.array_equal(ops.pack16_sorted(recs), np.unique(want_r[want_ok]))
        d = cuda(recs, torch.uint8)
        dr, dok = bd.pack16(d)
        assert np.array_equal(host(dok), want_ok) and np.array_equal(host(dr)[want_ok], want_r[want_ok])
        assert np.array_equal(host(bd.pack16_sorted(d)), np.unique(want_r[want_ok]))


@gpu
def test_pack16_sorted_duplicates_and_all_invalid(claimed):
    rng = np.random.default_rng(7)
    for n in PACK_SIZES[:-1]:
        recs = random_records(rng, n)
        recs = np.concatenate([recs, recs[rng.integers(0, n, n)]])              # every record again, some many times
        want_r, want_ok = ref_pack16(recs)
        assert np.array_equal(ops.pack16_sorted(recs), np.unique(want_r[want_ok]))
        assert np.array_equal(host(bd.pack16_sorted(cuda(recs, torch.uint8))), np.unique(want_r[want_ok]))
        junk = recs.copy()
        junk[:, rng.integers(0, 16)] = ord("N")                                  # all invalid
        assert ops.pack16_sorted(junk).size == 0 and bd.pack16_sorted(cuda(junk, torch.uint8)).numel() == 0
        assert not ops.pack16(junk)[1].any()


# ================================================================================================= 4. guard bands on caller outputs
PAD_BYTES = 4096
SENTINEL = {torch.int32: -0x5A5A1235, torch.uint8: 0xA7, torch.int64: -0x1234567890ABCDF}


class Guarded:
    """A caller buffer of n elements inside a larger tensor filled with a sentinel; the interior starts PAD_BYTES (a multiple of
    16) after the allocation, so every alignment check passes."""

    def __init__(self, n, dtype):
        self.pad = PAD_BYTES // torch.empty(0, dtype=dtype).element_size()
        self.n = n
        self.buf = torch.full((n + 2 * self.pad,), SENTINEL[dtype], dtype=dtype, device=bd._device())
        self.t = self.buf[self.pad:self.pad + n]

    @property
    def ptr(self):
        return self.t.data_ptr()

    def intact(self):
        s = SENTINEL[self.buf.dtype]
        return bool((self.buf[:self.pad] == s).all()) and bool((self.buf[self.pad + self.n:] == s).all())


def assert_guards(*gs):
    torch.cuda.synchronize()
    for g in gs:
        assert g.intact(), "a write landed outside the caller's buffer"


def check(rc):
    badger_b200._lib.check(rc)


@gpu
@pytest.mark.parametrize("n", PACK_SIZES)
def test_guard_bands_pack16_dedup_fetch_assign(n, pack_pool, claimed):
    L, st = badger_b200.lib(), bd._stream()
    recs = cuda(pack_pool[4096 - min(n, 4096) // 2:][:n], torch.uint8)
    out, val = Guarded(n, torch.int32), Guarded(n, torch.uint8)
    check(L.bdg_dev_pack16(recs.data_ptr(), n, out.ptr, val.ptr, st))
    assert_guards(out, val)                                   # before any unguarded call: a stray write lands in a band first
    want_r, want_ok = bd.pack16(recs)
    assert torch.equal(val.t.bool(), want_ok) and torch.equal(out.t[want_ok], want_r[want_ok])
    srt, k = Guarded(n, torch.int32), C.c_size_t(0)
    check(L.bdg_dev_pack16_sorted(recs.data_ptr(), n, srt.ptr, C.byref(k), st))
    assert_guards(srt)
    want_s = bd.pack16_sorted(recs)
    assert k.value == want_s.numel() and torch.equal(srt.t[:k.value], want_s)
    # the read map of n reads (distinct barcodes from a pool of about n / 3, every 7th row invalid) and its per-read gather
    rng = np.random.default_rng(n)
    keys = rng.integers(0, 1 << 32, max(n // 3, 1), dtype=np.uint64).astype(np.uint32)
    keys[:2] = [0, 0xFFFFFFFF][:keys.size]
    ranks = keys[rng.integers(0, keys.size, n)]
    valid = np.arange(n) % 7 != 3
    for mask in (None, valid):
        rm = bd.dedup_reads(cuda(ranks), None if mask is None else cuda(mask, torch.bool))
        N = rm.n_distinct
        want = {k: getattr(rm, k) for k in ("distinct", "counts", "sorted_pos", "sorted_distinct")}
        gs = [Guarded(N, torch.int32) for _ in range(4)]
        check(L.bdg_dev_dedup_fetch(rm.token, *[g.ptr for g in gs], st))
        assert_guards(*gs)
        for g, k in zip(gs, want):
            assert torch.equal(g.t.to(torch.int64) if k in ("counts", "sorted_pos") else g.t.view(want[k].dtype), want[k]), k
        ci = torch.from_numpy(rng.integers(-2, N, N).astype(np.int32)).to(bd._device())
        cen, has, m = Guarded(n, torch.int32), Guarded(n, torch.uint8), C.c_size_t(0)
        check(L.bdg_dev_assign_reads32(rm.token, ci.data_ptr(), N, cen.ptr, has.ptr, n, C.byref(m), st))
        assert_guards(cen, has)
        # plain restatement of the gather: row -> its distinct barcode -> its node -> the node's centre
        v = np.ones(n, bool) if mask is None else mask
        s_host = host(want["sorted_distinct"])
        node = np.minimum(np.searchsorted(s_host, ranks), N - 1)      # exact on valid rows; a barcode seen only in invalid rows is no node
        c = ci.cpu().numpy()
        ok = v & (c[node] >= 0)
        assert np.array_equal(host(has.t).astype(bool), ok)
        assert np.array_equal(host(cen.t)[ok], s_host[c[node[ok]]]) and m.value == int(ok.sum())


@gpu
@pytest.mark.parametrize("n", [2, 3, 255, 257, 1025, 4097, 70001])
def test_guard_bands_edges_build_and_copy(n, claimed):
    L, st = badger_b200.lib(), bd._stream()
    rng = synth.rng_for(n)
    cells = rng.integers(0, 1 << 32, max(n // 40, 1), dtype=np.uint64).astype(np.uint32)
    obs, _ = synth.simulate_reads(cells, 4 * n, 0.06, rng)
    s = synth.sorted_unique(np.concatenate([synth.sorted_unique(obs)[:n - 1], [0xFFFFFFFF]]))
    want = ops.canonical(*ops.edges_build(s, 2))
    E = want[0].size
    d_s = cuda(s)
    for cap in sorted({E, max(E - 1, 0)}):
        a, b, d = Guarded(cap, torch.int32), Guarded(cap, torch.int32), Guarded(cap, torch.uint8)
        cnt = Guarded(1, torch.int64)
        check(L.bdg_dev_edges_build(d_s.data_ptr(), s.size, 2, 0, 1, a.ptr if cap else None, b.ptr if cap else None,
                                    d.ptr if cap else None, cap, cnt.ptr, st))
        assert_guards(a, b, d, cnt)
        assert int(cnt.t.item()) == E
        if cap == E:
            got = ops.canonical(host(a.t), host(b.t), host(d.t))
            assert all(np.array_equal(x, y) for x, y in zip(got, want))
    for devs in contexts():
        badger_b200.init(devs)
        h = ops.edges_handle(s, 2)
        try:
            assert h.count == E
            a, b, d = Guarded(E, torch.int32), Guarded(E, torch.int32), Guarded(E, torch.uint8)
            check(badger_b200.lib().bdg_dev_edges_copy(h._h, a.ptr if E else None, b.ptr if E else None, d.ptr if E else None,
                                                       bd._stream()))
            assert_guards(a, b, d)
            got = ops.canonical(host(a.t), host(b.t), host(d.t))
            assert all(np.array_equal(x, y) for x, y in zip(got, want))
        finally:
            h.free()
