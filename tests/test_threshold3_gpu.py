"""Edge construction at t = 3 by the join form (bdg_join.cuh) against the CPU oracle: forced with bdg_set_edge_mode(2) and
BDG_JOIN3_MIN_N=0 so that small inputs take it too."""
import os

import numpy as np
import pytest

import badger_b200
from badger_b200 import ops, synth
from oracle import oracle as orc

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def join3(monkeypatch):
    monkeypatch.setenv("BDG_JOIN3_MIN_N", "0")
    assert badger_b200.init() >= 1
    L = badger_b200.lib()
    badger_b200._lib.check(L.bdg_set_edge_mode(2))
    yield
    badger_b200._lib.check(L.bdg_set_edge_mode(-1))


def edge_rows(a, b, d):
    a, b, d = ops.canonical(a, b, d)
    return np.stack([a, b, d], 1).astype(np.int64)


def oracle_rows(wa, wb, wd):
    return np.stack([wa, wb, wd], 1).astype(np.int64)


def clustered_set(seed, n_cells, reads, perr):
    rng = synth.rng_for(seed)
    cells = rng.integers(0, 1 << 32, n_cells, dtype=np.uint64).astype(np.uint32)
    obs, _ = synth.simulate_reads(cells, reads, perr, rng)
    return np.unique(obs)


def structured_set(rng, kind, n):
    """Small sets that stress the buckets, the candidate queues and the hand-over (the kinds of the t = 1 / 2 parity tests)."""
    if kind == 0:
        v = rng.integers(0, 1 << 32, n, dtype=np.uint64)
    elif kind == 1:
        v = np.arange(n, dtype=np.uint64) + np.uint64(int(rng.integers(0, (1 << 32) - n)))
    elif kind == 2:
        cells = rng.integers(0, 1 << 32, max(2, n // 40), dtype=np.uint64).astype(np.uint32)
        v, _ = synth.simulate_reads(cells, n, 0.10, rng, star_frac=0.0)
        v = v.astype(np.uint64)
    elif kind == 3:
        mask = [np.uint64(0xFFFF0000), np.uint64(0x0000FFFF), np.uint64(0x00FFFF00)][int(rng.integers(0, 3))]
        v = (rng.integers(0, 1 << 32, n, dtype=np.uint64) & ~mask) | (np.uint64(int(rng.integers(0, 1 << 32))) & mask)
    elif kind == 4:
        out = []
        for _ in range(n):
            unit = int(rng.integers(0, 1 << (2 * int(rng.integers(1, 4)))))
            ul = int(rng.integers(1, 4))
            w = 0
            for i in range(16):
                w |= ((unit >> (2 * (i % ul))) & 3) << (2 * i)
            for _e in range(int(rng.integers(0, 4))):
                w ^= int(rng.integers(1, 4)) << (2 * int(rng.integers(0, 16)))
            out.append(w)
        v = np.asarray(out, dtype=np.uint64)
    else:
        base = np.asarray([0, 1, 2, 3, 0xFFFFFFFF, 0xFFFFFFFE, 0x3FFFFFFF, 0x40000000, 0x7FFFFFFF, 0x80000000, 0xBFFFFFFF, 0xC0000000,
                           0x000FFFFF, 0x00100000, 0x0000FFFF, 0x00010000, 0x003FFFFF, 0x00400000], dtype=np.uint64)
        v = np.concatenate([base, base ^ np.uint64(0x55555555), rng.integers(0, 1 << 32, n, dtype=np.uint64)])
    return np.unique(v.astype(np.uint32))


@pytest.mark.parametrize("seed", [43, 44])
def test_join3_clustered_vs_oracle(seed):
    s = clustered_set(seed, 300, 8000, 0.08)
    a, b, d = ops.edges_build(s, 3)
    wa, wb, wd, _ = orc.Index(s).edges(3)
    assert np.array_equal(edge_rows(a, b, d), oracle_rows(wa, wb, wd))
    assert (d == 3).sum() > 100


def test_join3_structured_sets_vs_brute_force():
    rng = np.random.default_rng(303)
    total = 0
    for trial in range(24):
        kind = trial % 6
        n = int(rng.integers(2, 1200)) if trial % 5 else int(rng.integers(1200, 2500))
        s = structured_set(rng, kind, n)
        a, b, d = ops.edges_build(s, 3)
        wa, wb, wd = orc.edges_brute(s, 3)
        assert np.array_equal(edge_rows(a, b, d), oracle_rows(wa, wb, wd)), (trial, kind, s.size)
        total += a.size
    assert total > 10000


def test_join3_edge_cases():
    for arr in ([], [7], [0, 0xFFFFFFFF], [0, 1, 2, 3], list(range(2047, 2047 + 5)), list(range(100, 400))):
        s = np.asarray(arr, np.uint32)
        a, b, d = ops.edges_build(s, 3)
        wa, wb, wd = orc.edges_brute(s, 3)
        assert np.array_equal(edge_rows(a, b, d), oracle_rows(wa, wb, wd)), arr


def test_join3_edge_buffer_regrow(monkeypatch):
    s = clustered_set(55, 40, 20000, 0.06)
    want = edge_rows(*ops.edges_build(s, 3))
    assert want.shape[0] > (1 << 16) + 1024 + s.size
    badger_b200.lib().bdg_shutdown()
    monkeypatch.setenv("BDG_EDGE_CAP_PER_ROW", "1")
    badger_b200.init()
    badger_b200._lib.check(badger_b200.lib().bdg_set_edge_mode(2))
    got = edge_rows(*ops.edges_build(s, 3))
    assert np.array_equal(got, want)


@pytest.mark.parametrize("nparts", [1, 2, 3, 8])
def test_join3_parts_union_equals_full(nparts):
    """ops.edges_build_part is the streaming form (bdg_edges_build_into); the parts' union is the resident result."""
    s = clustered_set(77, 200, 12000, 0.08)
    full = edge_rows(*ops.edges_build(s, 3))
    merged = np.concatenate([edge_rows(*ops.edges_build_part(s, 3, p, nparts)) for p in range(nparts)])
    merged = merged[np.lexsort((merged[:, 1], merged[:, 0]))]
    assert np.array_equal(merged, full) and full.shape[0] > 1000


def test_join3_packed_pipeline_on_all_devices_matches_one_device():
    from badger_b200 import pipeline
    n_dev = badger_b200.init()
    many_devs = None if n_dev >= 2 else [0, 0]
    rng = synth.rng_for(124)
    wl = synth.make_whitelist(20000, rng)
    cells = synth.pick_cells(wl, 600, rng)
    obs, valid = synth.simulate_reads(cells, 80000, 0.08, rng)
    wls = np.sort(wl)
    res = []
    try:
        for devs in ([0], many_devs):
            badger_b200.init(devs)
            badger_b200._lib.check(badger_b200.lib().bdg_set_edge_mode(2))
            out, info = pipeline.assign_packed(obs, valid, threshold=3, n_cells=600, whitelist_sorted=wls)
            res.append((out, info))
    finally:
        badger_b200.init()
    assert np.array_equal(res[0][0], res[1][0]) and res[0][1] == res[1][1]
    assert res[0][1]["edges"] > 1000


def test_join3_graphs_golden(gold_graphs):
    from badger_b200 import BarcodeGraph
    n = 0
    for g in gold_graphs:
        if g["t"] != 3:
            continue
        bg = BarcodeGraph(g["t"])
        bg.graph_construction(g["reads"], 16, 1)
        a, b, d = bg.edge_arrays()
        assert np.stack([a, b, d], 1).astype(np.int64).tolist() == g["edges"], g["name"]
        n += 1
    assert n >= 1


def test_join3_full_size_sampled_rows():
    """A C4-sized synthetic set (2e7 reads, 4.6e6 distinct) at t = 3 on the default route (the join form): 1 500 sampled rows
    as either end point against the oracle's index walk, plus size-independent properties."""
    badger_b200._lib.check(badger_b200.lib().bdg_set_edge_mode(-1))
    os.environ.pop("BDG_JOIN3_MIN_N", None)
    workers = min(32, len(os.sched_getaffinity(0)))
    wl, cells, obs, valid, cfg = synth.make_dataset("C4", workers=workers)
    s = synth.sorted_unique(obs[valid])
    del obs, valid
    a, b, d = ops.edges_build(s, 3)
    assert a.size > 20 * s.size
    assert (a < b).all() and ((d >= 1) & (d <= 3)).all() and (d == 3).any()
    rows = np.sort(np.random.default_rng(13).choice(s.size, 1500, replace=False)).astype(np.uint32)
    wa, wb, wd = orc.edges_touching(orc.Index(s), 3, rows)
    picked = np.zeros(s.size, bool)
    picked[rows] = True
    sel = picked[np.searchsorted(s, a)] | picked[np.searchsorted(s, b)]
    assert np.array_equal(edge_rows(a[sel], b[sel], d[sel]), oracle_rows(wa, wb, wd))
    assert wa.size > rows.size
    part = (a & np.uint32(63)) == 7                               # no edge twice
    key = (a[part].astype(np.uint64) << np.uint64(32)) | b[part].astype(np.uint64)
    assert np.unique(key).size == key.size
