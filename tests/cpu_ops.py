"""Oracle-backed stand-ins for badger_b200.ops, used ONLY by the CPU (`not gpu`) tests to exercise the
host-side logic of the Python layer (centre selection, clustering, assignment, output) without a GPU."""
import numpy as np

from badger_b200 import synth
from oracle import oracle as orc


def pack16(seqs):
    if isinstance(seqs, np.ndarray):
        seqs = np.ascontiguousarray(seqs, dtype=np.uint8).tobytes()
    if isinstance(seqs, (bytes, bytearray)):
        seqs = [bytes(seqs[i:i + 16]) for i in range(0, len(seqs), 16)]
    out = np.zeros(len(seqs), np.uint32); valid = np.ones(len(seqs), bool)
    for i, s in enumerate(seqs):
        s = s.decode() if isinstance(s, bytes) else s
        try:
            out[i] = orc.rank(s)
        except KeyError:
            valid[i] = False
    return out, valid


def edges_build(sorted_unique, t):
    s = np.ascontiguousarray(sorted_unique, dtype=np.uint32)
    if s.size < 2 or t <= 0:
        return np.empty(0, np.uint32), np.empty(0, np.uint32), np.empty(0, np.uint8)
    a, b, d, _ = orc.Index(s).edges(t)
    return a, b, d


def edges_build_part(sorted_unique, t, part, nparts):
    from badger_b200.parallel import part_rows
    s = np.ascontiguousarray(sorted_unique, dtype=np.uint32)
    rows = part_rows(s.size, part, nparts)
    if s.size < 2 or t <= 0 or rows.size == 0:
        return np.empty(0, np.uint32), np.empty(0, np.uint32), np.empty(0, np.uint8)
    a, b, d, _ = orc.Index(s).edges(t, rows=rows)
    return a, b, d


def member_sorted(wl, q):
    return orc.member(wl, q).astype(bool)


def nearest_bounded(q, targets, max_d=2):
    return orc.nearest(q, targets, max_d)


def kmer_score(q, wl, min_kmers=1, cap=None):
    cnt, mult = orc.kmer_score(q, wl)
    qi, wi = np.nonzero((cnt >= max(min_kmers, 1)))
    return qi.astype(np.uint32), wi.astype(np.uint32), cnt[qi, wi], mult[qi, wi]


class KmerIndex:
    def __init__(self, known):
        self.known = np.ascontiguousarray(known, dtype=np.uint32)
        self.size = int(self.known.size)

    def query(self, q, min_kmers=1, cap=None):
        return kmer_score(q, self.known, min_kmers, cap)

    def free(self):
        pass


def dedup_first_seen(ranks, want_map=False, want_sorted_pos=False):
    r, c = orc.dedup_count(np.ascontiguousarray(ranks, dtype=np.uint32))
    out = (r, c.astype(np.int64))
    if want_map:
        pos = {int(v): i for i, v in enumerate(r.tolist())}
        out += (np.asarray([pos[int(v)] for v in np.asarray(ranks).tolist()], np.uint32),)
    if want_sorted_pos:
        out += (np.argsort(np.argsort(r, kind="stable"), kind="stable").astype(np.uint32),)
    return out


class ReadMap:
    """Stand-in for ops.ReadMap: everything the device would keep, as host arrays."""

    def __init__(self, distinct, counts, sorted_pos, n_valid, rows, token):
        self.distinct, self.counts, self.sorted_pos = distinct, counts, sorted_pos
        self.n_distinct, self.n_valid, self.rows, self.token = int(distinct.size), n_valid, rows, token
        s = np.empty_like(distinct)
        s[sorted_pos] = distinct
        self.sorted_distinct = s
        self.ci = None                                 # clustering left "on the device" by EdgeHandle.cluster_resident


def dedup_reads(ranks, valid=None):
    r = np.ascontiguousarray(ranks, dtype=np.uint32)
    v = np.ones(r.size, bool) if valid is None else np.asarray(valid, bool)
    if not v.any():
        return ReadMap(np.empty(0, np.uint32), np.empty(0, np.int64), np.empty(0, np.uint32), 0, int(r.size), 0)
    d, c, rmap, spos = dedup_first_seen(r[v], want_map=True, want_sorted_pos=True)
    rm = ReadMap(d, c, spos, int(v.sum()), int(r.size), 1)
    rm._cpu = (v, rmap)
    return rm


def assign_reads(rm, centre_idx):
    from badger_b200 import ops
    c32, has, n = assign_reads32(rm, centre_idx)
    return ops.widen(c32, has), n


def assign_reads32(rm, centre_idx=None):
    out = np.zeros(rm.rows, np.uint32); has = np.zeros(rm.rows, np.uint8)
    if rm.token == 0:
        return out, has, 0
    if centre_idx is None:
        centre_idx = _RESIDENT["ci"]
    v, rmap = rm._cpu
    s = rm.sorted_distinct
    ci = np.asarray(centre_idx, np.int32)[rm.sorted_pos]
    ok = ci >= 0
    cd = np.where(ok, s[np.maximum(ci, 0)], 0).astype(np.uint32)
    out[v] = cd[rmap]
    has[v] = ok[rmap]
    return out, has, int(has.sum())


_RESIDENT = {"ci": None}


def centres_above(rm, n_cells, whitelist_sorted=None):
    """barcode_graph.py:252-258 restated on the host arrays (the GPU operator's contract)."""
    first = rm.counts[:n_cells]
    cutoff = max((int(first.sum()) / first.size) / 5.0, 5)
    above = np.nonzero(rm.counts > cutoff)[0]
    above = above[np.argsort(-rm.counts[above], kind="stable")]
    top = rm.distinct[above]
    hits = None
    if whitelist_sorted is not None:
        hits = member_sorted(np.ascontiguousarray(whitelist_sorted, dtype=np.uint32), top) if top.size else np.zeros(0, bool)
    return float(cutoff), top, rm.counts[above], hits


def centres_rest(rm, cutoff, need):
    from badger_b200.barcode_graph import rest_by_counts
    return rest_by_counts(rm.distinct, rm.counts, cutoff, need - 1)[:need]


def pack16_sorted(records):
    r, ok = pack16(records)
    return np.unique(r[ok])


def cluster_levels(sorted_unique, ea, eb, centres, rounds=2, want_has_edge=False):
    """Literal restatement of the reference's rounds (oracle.cluster) turned into the operator's array form."""
    if want_has_edge:
        ci, lv = cluster_levels(sorted_unique, ea, eb, centres, rounds)
        s = np.ascontiguousarray(sorted_unique, dtype=np.uint32)
        has = np.zeros(s.size, bool)
        has[np.searchsorted(s, np.asarray(ea, np.uint32))] = True
        has[np.searchsorted(s, np.asarray(eb, np.uint32))] = True
        return ci, lv, has & (lv != 0)
    assert rounds == 2
    s = np.ascontiguousarray(sorted_unique, dtype=np.uint32)
    adj = {}
    for x, y in zip(np.asarray(ea).tolist(), np.asarray(eb).tolist()):
        adj.setdefault(int(x), []).append(int(y)); adj.setdefault(int(y), []).append(int(x))
    res = orc.cluster(adj, [int(c) for c in np.asarray(centres).tolist()])
    ci = np.full(s.size, -2, np.int32); lv = np.full(s.size, 255, np.uint8)
    pos = {int(v): i for i, v in enumerate(s.tolist())}
    for node, (cen, level) in res.items():
        if node not in pos:
            continue                                   # a centre that was never observed has no node
        if cen == -1:
            ci[pos[node]] = -1
        else:
            ci[pos[node]] = pos[cen]; lv[pos[node]] = level
    return ci, lv


class EdgeHandle:
    """Stand-in for ops.EdgeHandle (edges kept 'on the device')."""

    def __init__(self, s, t):
        self.s = s
        self.a, self.b, self.d = edges_build(s, t)
        self.count, self.n_nodes = int(self.a.size), int(s.size)

    def copy(self):
        return self.a, self.b, self.d

    def cluster_levels(self, centres, rounds=2, want_has_edge=False):
        return cluster_levels(self.s, self.a, self.b, centres, rounds, want_has_edge)

    def cluster_resident(self, centres, rounds=2):
        ci, lv, has_edge = cluster_levels(self.s, self.a, self.b, centres, rounds, True)
        _RESIDENT["ci"] = ci
        return int(has_edge.sum())

    def free(self):
        pass


def edges_handle(sorted_unique, t):
    return EdgeHandle(np.ascontiguousarray(sorted_unique, dtype=np.uint32), t)


def edges_handle_resident(rm, t):
    return EdgeHandle(np.ascontiguousarray(rm.sorted_distinct, dtype=np.uint32), t)


def install(monkeypatch):
    from badger_b200 import ops
    for name in ("pack16", "edges_build", "edges_build_part", "member_sorted", "nearest_bounded", "kmer_score", "dedup_first_seen",
                 "cluster_levels", "KmerIndex", "edges_handle", "edges_handle_resident", "dedup_reads", "assign_reads", "assign_reads32", "centres_above", "centres_rest",
                 "pack16_sorted"):
        monkeypatch.setattr(ops, name, globals()[name])
