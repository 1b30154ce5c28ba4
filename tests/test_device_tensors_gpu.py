"""badger_b200.device, the correction step on CUDA tensors, against the host operators and pipeline.assign_packed(form="u32"):
the same kernels behind device-pointer entry points, so every result must be equal element for element."""
import ctypes as C
import glob
import json
import os

import numpy as np
import pytest
import torch

import badger_b200
from badger_b200 import device as bd
from badger_b200 import ops, pipeline, synth
from gpu_helpers import claimed, cuda, dataset, host

pytestmark = [pytest.mark.gpu, pytest.mark.usefixtures("claimed")]


def assert_same_assignment(dev_out, host_out):
    (centre, has), info = dev_out
    (c32, h8), want_info = host_out
    assert centre.dtype in bd.BARCODE_DTYPES and has.dtype == torch.bool
    assert np.array_equal(host(centre), c32) and np.array_equal(host(has), h8.astype(bool))
    assert info == want_info


CASES = [  # threshold, whitelist, valid mask, true barcodes, high_sens, barcode dtype
    (1, True, True, False, False, torch.int32),
    (2, False, False, False, False, torch.uint32),
    (2, True, True, False, True, torch.int32),
    (2, False, True, True, True, torch.int32),
    (3, True, True, False, False, torch.uint32),
    (3, False, True, True, False, torch.int32),
]


@pytest.mark.parametrize("t,use_wl,use_valid,use_tb,high_sens,dtype", CASES)
def test_assign_packed_matches_host(t, use_wl, use_valid, use_tb, high_sens, dtype):
    wl, cells, obs, valid = dataset(500 + t, 200000 if t < 3 else 120000)
    assert not valid.all()
    wls = np.sort(wl)
    kw = dict(threshold=t, n_cells=600, high_sens=high_sens)
    tb = cells[:500].tolist() if use_tb else None
    want = pipeline.assign_packed(obs, valid if use_valid else None, whitelist_sorted=wls if use_wl else None, true_barcodes=tb,
                                  form="u32", **kw)
    got = bd.assign_packed(cuda(obs, dtype), cuda(valid, torch.bool) if use_valid else None,
                           whitelist_sorted=cuda(wls, dtype) if use_wl else None,
                           true_barcodes=cuda(cells[:500], dtype) if use_tb else None, **kw)
    assert got[0][0].dtype == dtype
    assert_same_assignment(got, want)
    assert want[1]["assigned_reads"] > want[1]["valid_reads"] // 2 and want[1]["edges"] > 1000


def test_assign_packed_edge_cases():
    (c, h), info = bd.assign_packed(torch.empty(0, dtype=torch.int32, device=bd._device()), threshold=1, n_cells=10)
    assert c.numel() == 0 and info == {"reads": 0, "valid_reads": 0}
    r = torch.arange(5, dtype=torch.int32, device=bd._device())
    (c, h), info = bd.assign_packed(r, torch.zeros(5, dtype=torch.uint8, device=bd._device()), threshold=1, n_cells=10)
    assert not h.any() and info["valid_reads"] == 0


def test_assign_packed_on_two_contexts_matches_one():
    """init([0, 0]) when the box has one GPU (two contexts on the same device), every device otherwise."""
    n_dev = badger_b200.init()
    many = None if n_dev >= 2 else [0, 0]
    wl, cells, obs, valid = dataset(611, 300000)
    wls = np.sort(wl)
    for t in (2, 3):
        res = []
        for devs in ([0], many):
            badger_b200.init(devs)
            got = bd.assign_packed(cuda(obs), cuda(valid, torch.bool), threshold=t, n_cells=600, whitelist_sorted=cuda(wls))
            want = pipeline.assign_packed(obs, valid, threshold=t, n_cells=600, whitelist_sorted=wls, form="u32")
            assert_same_assignment(got, want)
            res.append((host(got[0][0]), host(got[0][1]), got[1]))
        assert np.array_equal(res[0][0], res[1][0]) and np.array_equal(res[0][1], res[1][1]) and res[0][2] == res[1][2]


def test_dedup_reads_and_fetch_match_host():
    _, _, obs, valid = dataset(7, 150000)
    for v in (None, valid):
        want = ops.dedup_reads(obs, v)
        w = {k: getattr(want, k).copy() for k in ("distinct", "counts", "sorted_pos", "sorted_distinct")}
        got = bd.dedup_reads(cuda(obs, torch.uint32), None if v is None else cuda(v.astype(np.uint8) * 3, torch.uint8))
        assert (got.n_distinct, got.n_valid, got.rows) == (want.n_distinct, want.n_valid, want.rows)
        assert got.distinct.dtype == torch.uint32 and got.counts.dtype == torch.int64
        for k in w:
            assert np.array_equal(host(getattr(got, k)).astype(np.int64), w[k].astype(np.int64)), k


def test_pack16_and_pack16_sorted_match_host():
    rng = synth.rng_for(31)
    wl = synth.make_whitelist(30000, rng)
    recs = np.frombuffer(b"".join(synth.unrank_many(wl).tolist()), np.uint8).reshape(-1, 16).copy()
    recs[::97, 5] = ord("N")                                   # records the packing must drop / mark invalid
    recs = np.concatenate([recs, recs[:1000]])                 # duplicates
    d_recs = torch.from_numpy(recs).to(bd._device())
    r, ok = bd.pack16(d_recs)
    wr, wok = ops.pack16(recs)
    assert np.array_equal(host(ok), wok) and np.array_equal(host(r)[wok], wr[wok])
    s = bd.pack16_sorted(d_recs)
    assert np.array_equal(host(s), ops.pack16_sorted(recs))


def edge_rows(a, b, d):
    a, b, d = ops.canonical(a, b, d)
    return np.stack([a, b, d], 1).astype(np.int64)


@pytest.mark.parametrize("t", [1, 2, 3])
def test_edges_match_host(t, monkeypatch):
    _, _, obs, valid = dataset(40 + t, 400000)
    s = np.unique(obs[valid])
    want = edge_rows(*ops.edges_build(s, t))
    got = bd.edges(cuda(s), t)
    assert got[0].dtype == torch.int32 and got[2].dtype == torch.uint8
    assert np.array_equal(edge_rows(*map(host, got)), want) and want.shape[0] > 10000
    # a first guess of one edge per row is too small: the build runs again with the exact size
    monkeypatch.setenv("BDG_EDGE_CAP_PER_ROW", "1")
    assert want.shape[0] > bd._edge_cap(s.size, t)
    got = bd.edges(cuda(s, torch.uint32), t)
    assert np.array_equal(edge_rows(*map(host, got)), want)


def test_edges_copy_of_a_multi_device_handle():
    n_dev = badger_b200.init()
    badger_b200.init(None if n_dev >= 2 else [0, 0])
    _, _, obs, valid = dataset(83, 300000)
    s = np.unique(obs[valid])
    h = ops.edges_handle(s, 2)
    try:
        want = edge_rows(*h.copy())
        got = bd.edges_copy(h)
    finally:
        h.free()
    assert np.array_equal(edge_rows(*map(host, got)), want) and want.shape[0] > 10000


def test_stream_order_without_synchronisation():
    """The inputs come from a kernel queued on a side stream behind a long sleep; the call runs under that stream and nobody
    synchronises: the library must wait for the kernel, and the outputs must be complete when read on that stream."""
    wl, _, obs, valid = dataset(95, 300000)
    wls = np.sort(wl)
    want = pipeline.assign_packed(obs, valid, threshold=2, n_cells=600, whitelist_sorted=wls, form="u32")
    key = 0x5A5A5A5A
    src = cuda(obs) ^ key                                      # the input, scrambled; unscrambled on the side stream
    d_valid, d_wl = cuda(valid, torch.bool), cuda(wls)
    torch.cuda.synchronize()
    side = torch.cuda.Stream(device=bd._device())
    with torch.cuda.stream(side):
        torch.cuda._sleep(200_000_000)                         # ~0.1 s of spinning before the input exists
        ranks = src ^ key
        got = bd.assign_packed(ranks, d_valid, threshold=2, n_cells=600, whitelist_sorted=d_wl)
        centre, has = got[0][0].cpu(), got[0][1].cpu()         # copies queued on the side stream
    assert_same_assignment(((centre, has), got[1]), want)


def memcpy_bytes(trace_dir):
    """HtoD + DtoH bytes of the copies in the chrome traces torch.profiler wrote to trace_dir."""
    total = 0
    for path in glob.glob(os.path.join(trace_dir, "*.json")):
        with open(path) as fh:
            for ev in json.load(fh).get("traceEvents", []):
                name = ev.get("name", "")
                if ev.get("cat") == "gpu_memcpy" and ("HtoD" in name or "DtoH" in name):
                    total += int(ev.get("args", {}).get("bytes", 0))
    return total


def test_nothing_per_read_crosses_pcie(tmp_path):
    from torch.profiler import ProfilerActivity, profile
    wl, _, obs, valid = dataset(123, 1000000)
    wls = np.sort(wl)
    moved = {}
    for R in (250000, 1000000):
        d_obs, d_valid, d_wl = cuda(obs[:R]), cuda(valid[:R], torch.bool), cuda(wls)
        for form in ("device", "host"):
            run = (lambda: bd.assign_packed(d_obs, d_valid, threshold=2, n_cells=600, whitelist_sorted=d_wl)) if form == "device" else \
                  (lambda: pipeline.assign_packed(obs[:R], valid[:R], threshold=2, n_cells=600, whitelist_sorted=wls, form="u32"))
            run()                                              # warm: first-use uploads (seed tables) are not per read
            torch.cuda.synchronize()
            out = tmp_path / ("%s_%d" % (form, R))
            out.mkdir()
            with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
                run()
                torch.cuda.synchronize()
            prof.export_chrome_trace(str(out / "trace.json"))
            moved[form, R] = memcpy_bytes(str(out))
    print("PCIe bytes:", moved)
    assert moved["host", 1000000] > 8 * 1000000                # the check sees the per-read copies of the host form
    assert moved["device", 1000000] < 1000000
    assert moved["device", 1000000] < 2 * moved["device", 250000] + 65536


def test_errors_leave_the_library_usable():
    _, _, obs, valid = dataset(3, 20000)
    d_obs = cuda(obs)
    with pytest.raises(ValueError):
        bd.dedup_reads(torch.from_numpy(obs.view(np.int32)))                       # CPU tensor
    with pytest.raises(ValueError):
        bd.dedup_reads(torch.stack([d_obs, d_obs], 1)[:, 0])                       # not contiguous
    with pytest.raises(TypeError):
        bd.dedup_reads(d_obs.to(torch.int64))                                      # wrong dtype
    with pytest.raises(TypeError):
        bd.dedup_reads(d_obs, cuda(valid, torch.bool).to(torch.float32))
    with pytest.raises(ValueError):
        bd.pack16(torch.zeros(10, 15, dtype=torch.uint8, device=bd._device()))
    if torch.cuda.device_count() >= 2:
        with pytest.raises(ValueError):
            bd.dedup_reads(d_obs.to("cuda:1"))                                      # not the first claimed device
    # the C ABI refuses host memory where it takes device pointers
    L = badger_b200.lib()
    n, nv, tok = C.c_size_t(0), C.c_size_t(0), C.c_ulonglong(0)
    rc = L.bdg_dev_dedup_reads(obs.ctypes.data, None, obs.size, C.byref(n), C.byref(nv), C.byref(tok), bd._stream())
    assert rc == badger_b200._lib.BDG_ERR_ARG
    old = bd.dedup_reads(d_obs, cuda(valid, torch.bool))
    new = bd.dedup_reads(d_obs)
    with pytest.raises(badger_b200.BadgerB200Error):
        old.distinct                                                               # stale token
    assert new.distinct.numel() == new.n_distinct
    (c, h), info = bd.assign_packed(d_obs, cuda(valid, torch.bool), threshold=1, n_cells=100)
    want = pipeline.assign_packed(obs, valid, threshold=1, n_cells=100, form="u32")
    assert_same_assignment(((c, h), info), want)
