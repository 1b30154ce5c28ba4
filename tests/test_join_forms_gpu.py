"""Every instantiation of the join kernel (bdg_join.cuh: join_kernel<T, RS> for T = 2, 3 and RS = 8, 32) against the CPU oracle.
The library picks RS from the bucket length (RS = 32 only from about 12.6 M distinct barcodes), so BDG_JOIN_RS forces each
row-slab size on small sets here, and bdg_set_edge_mode(2) with BDG_JOIN3_MIN_N=0 forces the join at both thresholds."""
import ctypes as C

import numpy as np
import pytest

import badger_b200
from badger_b200 import ops, synth
from oracle import oracle as orc

pytestmark = pytest.mark.gpu


@pytest.fixture(params=[8, 32], ids=["rs8", "rs32"])
def rs(request, monkeypatch):
    monkeypatch.setenv("BDG_JOIN_RS", str(request.param))
    monkeypatch.setenv("BDG_JOIN3_MIN_N", "0")
    assert badger_b200.init() >= 1
    L = badger_b200.lib()
    badger_b200._lib.check(L.bdg_set_edge_mode(2))
    yield request.param
    badger_b200._lib.check(L.bdg_set_edge_mode(-1))


def clustered_set(seed, n_cells, reads, perr):
    rng = synth.rng_for(seed)
    cells = rng.integers(0, 1 << 32, n_cells, dtype=np.uint64).astype(np.uint32)
    obs, _ = synth.simulate_reads(cells, reads, perr, rng)
    return np.unique(obs)


def edge_rows(a, b, d):
    a, b, d = ops.canonical(a, b, d)
    return np.stack([a, b, d], 1).astype(np.int64)


@pytest.mark.parametrize("t", [2, 3])
def test_join_resident_vs_oracle(rs, t):
    s = clustered_set(91 + t, 300, 12000, 0.08)
    wa, wb, wd, _ = orc.Index(s).edges(t)
    want = np.stack([wa, wb, wd], 1).astype(np.int64)
    assert np.array_equal(edge_rows(*ops.edges_build(s, t)), want)
    assert (want[:, 2] == t).sum() > 100


@pytest.mark.parametrize("t", [2, 3])
def test_join_streaming_parts_union_equals_resident(rs, t):
    """ops.edges_build_part is the streaming form (bdg_edges_build_into); the parts' union is the resident result."""
    s = clustered_set(95 + t, 200, 12000, 0.08)
    full = edge_rows(*ops.edges_build(s, t))
    for nparts in (1, 3):
        merged = np.concatenate([edge_rows(*ops.edges_build_part(s, t, p, nparts)) for p in range(nparts)])
        merged = merged[np.lexsort((merged[:, 1], merged[:, 0]))]
        assert np.array_equal(merged, full), nparts
    assert full.shape[0] > 1000


@pytest.mark.parametrize("t", [2, 3])
def test_join_counters(rs, t):
    """bdg_dev_edges_stats_raw after one device-buffer call on one device: edges <= owned and scored <= within distance t
    <= candidates <= pairs tested."""
    import torch
    s = clustered_set(99 + t, 300, 12000, 0.08)
    L = badger_b200.lib()
    dev = torch.device("cuda", torch.cuda.current_device())
    stream = torch.cuda.current_stream(dev)
    d_s = torch.from_numpy(s.view(np.int32)).to(dev)
    cap = 64 * s.size
    d_a = torch.empty(cap, dtype=torch.int32, device=dev)
    d_b = torch.empty(cap, dtype=torch.int32, device=dev)
    d_d = torch.empty(cap, dtype=torch.uint8, device=dev)
    cnt = torch.zeros(1, dtype=torch.int64, device=dev)
    badger_b200._lib.check(L.bdg_dev_edges_build(d_s.data_ptr(), s.size, t, 0, 1, d_a.data_ptr(), d_b.data_ptr(), d_d.data_ptr(), cap,
                                                 cnt.data_ptr(), stream.cuda_stream))
    raw = (C.c_ulonglong * 8)()
    badger_b200._lib.check(L.bdg_dev_edges_stats_raw(raw, stream.cuda_stream))
    n = int(cnt.item())
    assert 1000 < n <= cap
    assert n <= raw[7] <= raw[6] <= raw[3] <= raw[2]
    a = d_a[:n].cpu().numpy().view(np.uint32); b = d_b[:n].cpu().numpy().view(np.uint32); d = d_d[:n].cpu().numpy()
    assert np.array_equal(edge_rows(a, b, d), edge_rows(*ops.edges_build(s, t)))
