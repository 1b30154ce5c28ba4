"""The correction step over reads that arrive in batches (pipeline.Tally, device.Tally, bdg_tally_* / bdg_[dev_]assign_lookup32)
against the one-call step: whatever the batching of `add` and of `assign`, the per-read result and `info` must equal
pipeline.assign_packed(form="u32") over the concatenation of the added batches, element for element.

- Parity on the datasets and variants of the one-call tests: thresholds 1-3, whitelist or none, valid masks, true_barcodes, high_sens
  in the default and the "set" order, int32 / uint32, the numpy and the tensor form; one batch, even, uneven, empty and one-row
  batches, a batch without a valid row, barcodes first seen in the last batch.  One C4-shaped set against the oracle stand-ins.
- The merge at scale: C4 (2e7 reads) in 7 uneven batches gives the read-map arrays of one dedup call.
- Past the one-call limit: a batch made on the device is added K times, K * R > 2^31.
- The contracts of the new entry points: guard bands, stream order, what crosses PCIe, refusals each followed by a working call,
  two device contexts."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import badger_b200
import test_step_vs_oracle_gpu as sv
from badger_b200 import device as bd
from badger_b200 import ops, pipeline, synth
from badger_b200._lib import BDG_ERR_ARG, BadgerB200Error
from gpu_helpers import claimed, cuda, dataset, host

pytestmark = [pytest.mark.gpu, pytest.mark.usefixtures("claimed")]
TESTS = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(TESTS)


def cuts(R, kind, seed):
    """Batch boundaries [(start, end), ...] covering 0 .. R in order."""
    rng = np.random.default_rng(seed)
    if kind == "one":
        pts = []
    elif kind == "even":
        pts = [R * k // 7 for k in range(1, 7)]
    elif kind == "uneven":                                    # random cuts, two empty batches, two one-row batches, a tiny first batch
        pts = sorted(rng.integers(1, R, 9).tolist())
        a, b = int(rng.integers(2, R - 2)), int(rng.integers(2, R - 2))
        pts = sorted(pts + [a, a, b, b + 1, 3, 0, R])
    elif kind == "rows":                                      # many small batches
        pts = list(range(0, R, max(R // 40, 1)))
    else:
        raise ValueError(kind)
    pts = [0] + pts + [R]
    return list(zip(pts[:-1], pts[1:]))


def run_numpy(obs, valid, add_kind, assign_kind, seed, **kw):
    t = pipeline.Tally()
    try:
        for s, e in cuts(obs.size, add_kind, seed):
            t.add(obs[s:e], None if valid is None else valid[s:e])
        info = t.finish(**kw)
        parts = [t.assign(obs[s:e], None if valid is None else valid[s:e]) for s, e in cuts(obs.size, assign_kind, seed + 1)]
    finally:
        t.free()
    return (np.concatenate([p[0] for p in parts]), np.concatenate([p[1] for p in parts])), info


def run_tensor(d_obs, d_valid, add_kind, assign_kind, seed, **kw):
    t = bd.Tally()
    R = d_obs.numel()
    try:
        for s, e in cuts(R, add_kind, seed):
            t.add(d_obs[s:e], None if d_valid is None else d_valid[s:e])
        info = t.finish(**kw)
        parts = [t.assign(d_obs[s:e], None if d_valid is None else d_valid[s:e]) for s, e in cuts(R, assign_kind, seed + 1)]
    finally:
        t.free()
    return (torch.cat([p[0] for p in parts]), torch.cat([p[1] for p in parts])), info


def assert_same(got, want):
    (c, h), info = got
    (wc, wh), winfo = want
    if isinstance(c, torch.Tensor):
        assert h.dtype == torch.bool
        c, h = host(c), host(h)
    assert np.array_equal(np.asarray(h).astype(bool), wh.astype(bool))
    assert np.array_equal(np.asarray(c), wc)
    assert info == winfo


def first_seen_late(obs, valid, last_start):
    """Barcodes whose first valid sighting lies in the rows from last_start on."""
    v = np.ones(obs.size, bool) if valid is None else valid
    early = set(np.unique(obs[:last_start][v[:last_start]]).tolist())
    return len(set(np.unique(obs[last_start:][v[last_start:]]).tolist()) - early)


# ================================================================================================= 1. parity with the one-call step
CASES = [  # threshold, whitelist, valid mask, true barcodes, high_sens, centre_order, dtype, add batching, assign batching
    (1, True, True, False, False, None, torch.int32, "uneven", "even"),
    (2, False, False, False, False, None, torch.uint32, "even", "uneven"),
    (2, True, True, False, True, None, torch.int32, "uneven", "one"),
    (2, True, True, False, True, "set", torch.uint32, "rows", "uneven"),
    (2, False, True, True, True, None, torch.int32, "one", "rows"),
    (3, True, True, False, False, None, torch.uint32, "uneven", "uneven"),
    (3, False, True, True, False, None, torch.int32, "rows", "even"),
]


@pytest.mark.parametrize("t,use_wl,use_valid,use_tb,high_sens,order,dtype,add_kind,assign_kind", CASES)
def test_batches_match_one_call(t, use_wl, use_valid, use_tb, high_sens, order, dtype, add_kind, assign_kind):
    wls, cells, obs, valid = dataset(500 + t, 200000 if t < 3 else 120000)
    v = valid if use_valid else None
    kw = dict(threshold=t, n_cells=600, high_sens=high_sens, centre_order=order, whitelist_sorted=wls if use_wl else None,
              true_barcodes=cells[:500].tolist() if use_tb else None)
    want = pipeline.assign_packed(obs, v, form="u32", **kw)
    assert want[1]["assigned_reads"] > want[1]["valid_reads"] // 2 and want[1]["edges"] > 1000
    if add_kind != "one":
        last = [s for s, e in cuts(obs.size, add_kind, t) if e - s > 100][-1]
        assert first_seen_late(obs, v, last) > 0, "the last batch must bring barcodes of its own"
    assert_same(run_numpy(obs, v, add_kind, assign_kind, t, **kw), want)
    kw_dev = dict(kw, whitelist_sorted=cuda(wls, dtype) if use_wl else None, true_barcodes=cuda(cells[:500], dtype) if use_tb else None)
    got = run_tensor(cuda(obs, dtype), cuda(valid, torch.bool) if use_valid else None, add_kind, assign_kind, t, **kw_dev)
    assert got[0][0].dtype == dtype
    assert_same(got, want)


def test_empty_batches_and_a_batch_without_valid_rows():
    """An all-invalid stretch of rows in the middle gets a batch of its own; empty batches on both sides of it."""
    wls, _, obs, valid = dataset(77, 150000)
    junk = np.arange(5000, dtype=np.uint32) * np.uint32(2654435761)              # wraps modulo 2^32
    k = 70000
    obs2 = np.concatenate([obs[:k], junk, obs[k:]])
    valid2 = np.concatenate([valid[:k], np.zeros(junk.size, bool), valid[k:]])
    kw = dict(threshold=2, n_cells=600, whitelist_sorted=wls)
    want = pipeline.assign_packed(obs2, valid2, form="u32", **kw)
    bounds = [0, 0, k, k, k + junk.size, k + junk.size, obs2.size, obs2.size]
    for form in ("numpy", "tensor"):
        t = pipeline.Tally() if form == "numpy" else bd.Tally()
        x, m = (obs2, valid2) if form == "numpy" else (cuda(obs2), cuda(valid2, torch.bool))
        nvs = [t.add(x[s:e], m[s:e]) for s, e in zip(bounds[:-1], bounds[1:])]
        assert nvs[3] == 0 and nvs[0] == nvs[2] == 0 and sum(nvs) == want[1]["valid_reads"]
        info = t.finish(**dict(kw, whitelist_sorted=wls if form == "numpy" else cuda(wls)))
        c, h = t.assign(x, m)
        assert_same(((c, h), info), want)
        # rows without a valid barcode only, and no rows at all
        c, h = t.assign(x[k:k + junk.size], m[k:k + junk.size])
        assert not h.any()
        assert len(t.assign(x[:0], m[:0])[0]) == 0
        t.free()


def test_nothing_valid_at_all():
    for form in ("numpy", "tensor"):
        t = pipeline.Tally() if form == "numpy" else bd.Tally()
        r = np.arange(7, dtype=np.uint32)
        x, m = (r, np.zeros(7, bool)) if form == "numpy" else (cuda(r), cuda(np.zeros(7, bool), torch.bool))
        t.add(x, m)
        t.add(x[:0], m[:0])
        info = t.finish(threshold=1, n_cells=10)
        want = pipeline.assign_packed(r, np.zeros(7, bool), threshold=1, n_cells=10, form="u32")
        c, h = t.assign(x, m)
        assert_same(((c, h), info), want)
        with pytest.raises(ValueError):
            t.assign(x)                                       # valid rows, and nothing was counted
        t.free()


def test_c4_shaped_batches_match_the_oracle(monkeypatch):
    """C4 at 1e6 reads, t = 2, against the oracle stand-ins of tests/cpu_ops.py (the one-call step run through the oracle)."""
    name = "C4_t2"
    D = sv.step_data(name)
    for variant in ("whitelist", "high_sens"):
        want = sv.oracle_step(name, variant, monkeypatch)[:2]
        kw = sv.step_kwargs(name, variant)
        assert_same(run_numpy(D["obs"], D["valid"], "uneven", "even", 41, **kw), want)
        got = run_tensor(cuda(D["obs"]), cuda(D["valid"], torch.bool), "even", "uneven", 42,
                         **dict(kw, whitelist_sorted=cuda(kw["whitelist_sorted"])))
        assert_same(got, want)


# ================================================================================================= 2. the merge at scale
def finish_raw(t):
    n, nv, tok = C.c_size_t(0), C.c_size_t(0), C.c_ulonglong(0)
    sv.check(badger_b200.lib().bdg_dev_tally_finish(t._handle(), C.byref(n), C.byref(nv), C.byref(tok), bd._stream()))
    return ops.ReadMap(int(n.value), int(nv.value), 0, int(tok.value))


def read_map_arrays(rm):
    return {k: np.array(getattr(rm, k)) for k in ("distinct", "counts", "sorted_pos", "sorted_distinct")}


def test_c4_in_seven_uneven_batches_gives_the_dedup_of_the_whole():
    _, _, obs, valid, _ = synth.make_dataset("C4")
    R = obs.size
    pts = [0, 1, 3_000_000, 3_000_001, 9_500_000, 10_250_000, 17_000_000, R]     # 7 batches, one of one row
    t = bd.Tally()
    d_obs, d_valid = cuda(obs), cuda(valid, torch.bool)
    for s, e in zip(pts[:-1], pts[1:]):
        t.add(d_obs[s:e], d_valid[s:e])
    got = read_map_arrays(finish_raw(t))
    t.free()
    want = read_map_arrays(ops.dedup_reads(obs, valid))
    assert got["distinct"].size > 1_000_000
    for k in want:
        assert np.array_equal(got[k], want[k]), k


# ================================================================================================= 3. past the one-call limit
def test_more_than_2_31_reads():
    """One seeded batch of 1e8 rows made on the device (rows drawn from a 1e6-read dataset) is added 22 times: 2.2e9 > 2^31 rows.
    The counts are exactly 22x, the first-seen order is the batch's, and assigning the batch gives the one-batch result.  With
    true_barcodes the centres are those barcodes followed by the head of the count-descending order (ties by first sighting),
    and multiplying every count by 22 keeps that order, ties included: the centre selection, and so the clustering, cannot change."""
    wls, cells, obs, valid = dataset(909, 1_000_000)
    g = torch.Generator(device=bd._device())
    g.manual_seed(2026)
    R, K = 100_000_000, 22
    idx = torch.randint(0, obs.size, (R,), generator=g, device=bd._device())
    batch, bvalid = cuda(obs)[idx], cuda(valid, torch.bool)[idx]
    del idx
    kw = dict(threshold=2, n_cells=600, whitelist_sorted=cuda(wls), true_barcodes=cuda(cells[:500]))
    one = bd.Tally()
    one.add(batch, bvalid)
    info1 = one.finish(**kw)
    want = one.assign(batch, bvalid)
    rm1 = read_map_arrays(ops.ReadMap(info1["distinct"], info1["valid_reads"], 0, one._rm.token))
    one.free()
    many = bd.Tally()
    for _ in range(K):
        many.add(batch, bvalid)
    assert many.rows == K * R > 1 << 31
    rmK = read_map_arrays(finish_raw(many))
    assert np.array_equal(rmK["distinct"], rm1["distinct"]) and np.array_equal(rmK["counts"], K * rm1["counts"])
    assert np.array_equal(rmK["sorted_pos"], rm1["sorted_pos"]) and np.array_equal(rmK["sorted_distinct"], rm1["sorted_distinct"])
    infoK = many.finish(**kw)
    for k in range(2):                                        # every batch is the same rows: every assign gives the one-batch result
        c, h = many.assign(batch, bvalid)
        assert torch.equal(c, want[0]) and torch.equal(h, want[1])
    assert infoK == dict(info1, reads=K * R, valid_reads=K * info1["valid_reads"], assigned_reads=2 * info1["assigned_reads"])
    many.free()


def test_a_count_of_2_32_is_refused_at_finish():
    b = torch.full((1 << 28,), 0x1234567, dtype=torch.int32, device=bd._device())
    t = bd.Tally()
    for _ in range(15):
        t.add(b)
    t.add(b[:-1])
    t.finish(threshold=1, n_cells=1, true_barcodes=[0x1234567])          # 2^32 - 1: still a uint32 count
    t.free()
    t = bd.Tally()
    for _ in range(16):
        t.add(b)
    with pytest.raises(BadgerB200Error) as e:
        t.finish(threshold=1, n_cells=1)
    assert e.value.code == BDG_ERR_ARG
    t.free()
    del b
    small = pipeline.Tally()                                  # the library still works
    small.add(np.array([5, 5, 6], np.uint32))
    small.finish(threshold=1, n_cells=1, true_barcodes=[5])
    c, h = small.assign(np.array([6, 5], np.uint32))
    assert c[1] == 5 and h[1] == 1


# ================================================================================================= 4. contracts
def test_guard_bands_of_the_lookup():
    L, st = badger_b200.lib(), bd._stream()
    rng = np.random.default_rng(5)
    for n in (1, 255, 257, 1025, 70001):
        keys = rng.integers(0, 1 << 32, max(n // 3, 1), dtype=np.uint64).astype(np.uint32)
        keys[:2] = [0, 0xFFFFFFFF][:keys.size]
        ranks = keys[rng.integers(0, keys.size, n)]
        valid = np.arange(n) % 7 != 3
        t = bd.Tally()
        t.add(cuda(ranks), cuda(valid, torch.bool))
        rm = finish_raw(t)
        N = rm.n_distinct
        s_host = rm.sorted_distinct
        ci = torch.from_numpy(rng.integers(-2, N, N).astype(np.int32)).to(bd._device())
        cen, has, m, miss = sv.Guarded(n, torch.int32), sv.Guarded(n, torch.uint8), C.c_size_t(0), C.c_size_t(0)
        d_r, d_v = cuda(ranks), cuda(valid, torch.bool)
        sv.check(L.bdg_dev_assign_lookup32(rm.token, ci.data_ptr(), N, d_r.data_ptr(), d_v.data_ptr(), n, cen.ptr, has.ptr, C.byref(m),
                                           C.byref(miss), st))
        sv.assert_guards(cen, has)
        node = np.minimum(np.searchsorted(s_host, ranks), N - 1)
        found = s_host[node] == ranks
        c = ci.cpu().numpy()
        ok = valid & found & (c[node] >= 0)
        assert np.array_equal(host(has.t).astype(bool), ok)
        assert np.array_equal(host(cen.t)[ok], s_host[c[node[ok]]]) and m.value == int(ok.sum())
        assert miss.value == int((valid & ~found).sum())       # barcodes seen only in invalid rows are no nodes
        t.free()


def test_stream_order_without_synchronisation():
    wls, _, obs, valid = dataset(95, 300000)
    kw = dict(threshold=2, n_cells=600)
    want = pipeline.assign_packed(obs, valid, whitelist_sorted=wls, form="u32", **kw)
    key = 0x5A5A5A5A
    src = cuda(obs) ^ key
    d_valid, d_wl = cuda(valid, torch.bool), cuda(wls)
    torch.cuda.synchronize()
    side = torch.cuda.Stream(device=bd._device())
    t = bd.Tally()
    with torch.cuda.stream(side):
        torch.cuda._sleep(200_000_000)                         # ~0.1 s of spinning before the first batch exists
        ranks = src ^ key
        t.add(ranks[:100000], d_valid[:100000])
        torch.cuda._sleep(100_000_000)
        ranks2 = src ^ key
        t.add(ranks2[100000:], d_valid[100000:])
        info = t.finish(whitelist_sorted=d_wl, **kw)
        torch.cuda._sleep(200_000_000)
        ranks3 = src ^ key
        c, h = t.assign(ranks3, d_valid)
        c, h = c.cpu(), h.cpu()                                # copies queued on the side stream
    t.free()
    assert_same(((c, h), info), want)


def pcie_probe(out_dir):
    """HtoD + DtoH bytes of one add and one assign of R rows on tensors, at two sizes, and of one add of the numpy form (the
    control: there every row crosses PCIe).  Prints them as one JSON line."""
    from torch.profiler import ProfilerActivity, profile
    from test_device_tensors_gpu import memcpy_bytes
    badger_b200.init()
    wls, _, obs, valid = dataset(123, 1000000)
    d_obs, d_valid = cuda(obs), cuda(valid, torch.bool)
    moved = {}

    def traced(name, fn):
        fn()                                                   # warm: first-use allocations are not per read
        torch.cuda.synchronize()
        out = os.path.join(out_dir, name)
        os.mkdir(out)
        with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        prof.export_chrome_trace(os.path.join(out, "trace.json"))
        moved[name] = memcpy_bytes(out)

    for R in (250000, 1000000):
        t = bd.Tally()
        traced("add_%d" % R, lambda: t.add(d_obs[:R], d_valid[:R]))
        t.finish(threshold=2, n_cells=600, whitelist_sorted=cuda(wls))
        traced("assign_%d" % R, lambda: t.assign(d_obs[:R], d_valid[:R]))
        t.free()
    h = pipeline.Tally()
    traced("host_add_1000000", lambda: h.add(obs, valid))
    h.free()
    print(json.dumps(moved))


def test_only_sizes_cross_pcie_per_add_and_assign(tmp_path):
    """The profiler runs in a process of its own: a profiler session leaves state behind in the process that ran it (later traces
    there have been seen to miss copies), and the PCIe checks of the other test files run in this process."""
    code = "import sys; sys.path[:0] = %r; import test_batched_step_gpu as m; m.pcie_probe(%r)" % ([TESTS, ROOT], str(tmp_path))
    res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stderr[-4000:]
    moved = json.loads(res.stdout.strip().splitlines()[-1])
    print("PCIe bytes:", moved)
    assert moved["host_add_1000000"] > 4 * 1000000             # the check sees the per-read copies of the numpy form
    for what in ("add", "assign"):
        assert moved["%s_1000000" % what] < 4096 and moved["%s_250000" % what] < 4096


def test_refusals_each_followed_by_a_working_call():
    wls, _, obs, valid = dataset(3, 60000)
    kw = dict(threshold=1, n_cells=100)
    want = pipeline.assign_packed(obs, valid, form="u32", **kw)
    L, st = badger_b200.lib(), bd._stream()
    t = bd.Tally()
    d_obs, d_valid = cuda(obs), cuda(valid, torch.bool)
    with pytest.raises(ValueError):
        t.assign(d_obs, d_valid)                               # assign before finish
    n, m = C.c_size_t(0), C.c_size_t(0)
    out, hs = torch.empty_like(d_obs), torch.empty(obs.size, dtype=torch.uint8, device=bd._device())
    assert L.bdg_dev_assign_lookup32(0, None, 1, d_obs.data_ptr(), None, obs.size, out.data_ptr(), hs.data_ptr(), C.byref(n), C.byref(m), st) == BDG_ERR_ARG
    # a batch of 2^31 rows, host and device form: refused before any row is read
    assert L.bdg_dev_tally_add(t._handle(), d_obs.data_ptr(), None, 1 << 31, None, st) == BDG_ERR_ARG
    assert L.bdg_tally_add(t._handle(), obs.ctypes.data, None, 1 << 31, None) == BDG_ERR_ARG
    with pytest.raises(TypeError):
        t.add(d_obs.to(torch.int64))
    with pytest.raises(ValueError):
        t.add(d_obs, d_valid[:-1])
    assert L.bdg_dev_tally_add(t._handle(), obs.ctypes.data, None, obs.size, None, st) == BDG_ERR_ARG       # host memory
    t.add(d_obs[:30000], d_valid[:30000])
    t.add(d_obs[30000:], d_valid[30000:])
    info = t.finish(**kw)
    with pytest.raises(BadgerB200Error):
        t.add(d_obs, d_valid)                                  # add after finish
    bad = d_obs.clone()
    i = int(valid.argmax())
    bad[i] = bad[i] ^ 0x0F0F0F0F                               # a barcode no batch held
    assert not bool(torch.isin(bad[i], d_obs[d_valid]))
    with pytest.raises(ValueError):
        t.assign(bad, d_valid)                                 # n_missing > 0
    c, h = t.assign(d_obs, d_valid)                            # working call
    assert_same(((c, h), info), want)
    ops.dedup_reads(obs[:1000])                                # a foreign dedup kills the token
    with pytest.raises(BadgerB200Error):
        t.assign(d_obs, d_valid)
    info = t.finish(**kw)                                      # finish again installs the read map anew
    c, h = t.assign(d_obs, d_valid)
    assert_same(((c, h), info), want)
    t.free()
    with pytest.raises(ValueError):
        t.add(d_obs)                                           # freed


def test_two_device_contexts():
    n_dev = badger_b200.init()
    many = None if n_dev >= 2 else [0, 0]
    wls, _, obs, valid = dataset(611, 300000)
    kw = dict(threshold=2, n_cells=600, whitelist_sorted=wls)
    want = pipeline.assign_packed(obs, valid, form="u32", **kw)
    for devs in ([0], many):
        badger_b200.init(devs)
        assert_same(run_numpy(obs, valid, "uneven", "even", 8, **kw), want)
        got = run_tensor(cuda(obs), cuda(valid, torch.bool), "even", "uneven", 9, **dict(kw, whitelist_sorted=cuda(wls)))
        assert_same(got, want)
