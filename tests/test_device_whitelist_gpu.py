"""badger_b200.device's whitelist operators (member_sorted, nearest_bounded, kmer_score, KmerIndex) on CUDA tensors, against the
host operators of ops (the same kernels behind host-buffer entry points: equal element for element, hits after sorting them by
(query, string)) and, on a sample, against the oracle."""
import ctypes as C
import glob
import json
import os

import numpy as np
import pytest
import torch

import badger_b200
from badger_b200 import device as bd
from badger_b200 import ops, synth
from gpu_helpers import claimed, cuda, host
from oracle import oracle as orc

pytestmark = [pytest.mark.gpu, pytest.mark.usefixtures("claimed")]

LOW_COMPLEXITY = np.asarray([0, 0x55555555, 0xAAAAAAAA, 0xFFFFFFFF, 0x11111111, 0x1B1B1B1B, 0xE4E4E4E4, 0x0F0F0F0F], np.uint32)


def npy(t):
    return t.cpu().numpy()


def randu32(rng, n):
    return rng.integers(0, 1 << 32, n, dtype=np.uint64).astype(np.uint32)


def whitelist(rng, W):
    wl = np.unique(randu32(rng, W + W // 50 + 16))
    return np.sort(wl[rng.permutation(wl.size)[:W]])


def near_queries(rng, known, n, err=0.08):
    """Queries drawn around the known strings (substitutions, indels), plus a few strings of their own and the low-complexity words."""
    obs, _ = synth.simulate_reads(known[rng.integers(0, known.size, max(n // 50, 1))], n, err, rng)
    return np.concatenate([obs, randu32(rng, 40), LOW_COMPLEXITY])


def canonical_hits(hq, hw, cnt, pos):
    """Hits as numpy arrays sorted by (query, string); the order of the hits is unspecified."""
    hq, hw, cnt, pos = (host(x) if isinstance(x, torch.Tensor) else x for x in (hq, hw, cnt, pos))
    hq, hw = hq.astype(np.uint32), hw.astype(np.uint32)
    o = np.lexsort((hw, hq))
    return hq[o], hw[o], cnt[o], pos[o]


def assert_same_hits(got, want):
    g, w = canonical_hits(*got), canonical_hits(*want)
    for x, y, name in zip(g, w, ("hit_q", "hit_w", "cnt", "pos")):
        assert np.array_equal(x, y), name


def assert_hits_match_oracle(hits, q, wl, min_kmers, sample):
    """The hits of the sampled queries are exactly the oracle's (query, string) pairs with S >= min_kmers, with S and the per-position
    counts."""
    hq, hw, cnt, pos = canonical_hits(*hits)
    wc, wm = orc.kmer_score(q[sample], wl)
    for k, qi in enumerate(sample):
        sel = hq == qi
        ww = np.nonzero(wc[k] >= max(min_kmers, 1))[0]
        assert np.array_equal(hw[sel], ww) and np.array_equal(cnt[sel], wc[k, ww]) and np.array_equal(pos[sel], wm[k, ww])


# ---------------------------------------------------------------------------------------------------------- a-6 membership
def test_member_matches_host_at_whitelist_size():
    rng = synth.rng_for(61)
    wl = whitelist(rng, 3_000_000)
    q = np.concatenate([randu32(rng, 600_000), wl[rng.integers(0, wl.size, 400_000)], np.asarray([0, 0xFFFFFFFF], np.uint32)])
    q = q[rng.permutation(q.size)]
    want = ops.member_sorted(wl, q)
    for dtype in bd.BARCODE_DTYPES:
        got = bd.member_sorted(cuda(wl, dtype), cuda(q, dtype))
        assert got.dtype == torch.bool and got.shape == (q.size,)
        assert np.array_equal(host(got), want)
    assert 350_000 < want.sum() < 450_000
    assert np.array_equal(want[:5000], orc.member(wl, q[:5000]).astype(bool))


def test_member_edge_sizes():
    rng = synth.rng_for(62)
    q = np.concatenate([randu32(rng, 1000), np.asarray([0, 7, 0xFFFFFFFF], np.uint32)])
    for wl in (np.empty(0, np.uint32), np.asarray([7], np.uint32), np.asarray([0xFFFFFFFF], np.uint32)):
        got = host(bd.member_sorted(cuda(wl), cuda(q)))
        assert np.array_equal(got, ops.member_sorted(wl, q)) and np.array_equal(got, orc.member(wl, q).astype(bool))
    assert bd.member_sorted(cuda(np.asarray([1, 2], np.uint32)), cuda(np.empty(0, np.uint32))).numel() == 0


def test_member_refuses_an_unsorted_whitelist():
    rng = synth.rng_for(63)
    wl = whitelist(rng, 100_000)
    bad = wl.copy()
    bad[70_000], bad[70_001] = bad[70_001], bad[70_000]
    q = wl[:1000]
    with pytest.raises(badger_b200.BadgerB200Error) as host_err:
        ops.member_sorted(bad, q)
    with pytest.raises(badger_b200.BadgerB200Error) as dev_err:
        bd.member_sorted(cuda(bad), cuda(q))
    assert str(dev_err.value) == str(host_err.value) and "70001" in str(dev_err.value)
    assert dev_err.value.code == badger_b200._lib.BDG_ERR_ARG
    assert host(bd.member_sorted(cuda(wl), cuda(q))).all()          # a working call follows
    dup = np.sort(np.concatenate([wl, wl[:10]]))                      # repeated entries are sorted: accepted, as on the host
    assert np.array_equal(host(bd.member_sorted(cuda(dup), cuda(q))), ops.member_sorted(dup, q))


# ---------------------------------------------------------------------------------------------------------- a-7 nearest
def nearest_case(seed, n_q):
    """Targets with near-duplicates (ties on distance), exact duplicates and the extreme words, in a shuffled caller order."""
    rng = synth.rng_for(seed)
    centres = randu32(rng, 6000)
    obs, _ = synth.simulate_reads(centres, n_q, 0.07, rng)
    q = np.concatenate([obs, centres[:300], randu32(rng, 500), np.asarray([0, 0xFFFFFFFF, 0x55555555], np.uint32)])
    tg = np.concatenate([centres, centres[:200] ^ np.uint32(1), centres[:100], np.asarray([0, 0xFFFFFFFF], np.uint32)])
    return rng, q, tg[rng.permutation(tg.size)]


@pytest.mark.parametrize("max_d", [0, 1, 2, 3])
@pytest.mark.parametrize("n_q", [1500, 80_000])
def test_nearest_matches_host(max_d, n_q):
    rng, q, tg = nearest_case(70 + max_d, n_q)
    sparse = q.size * tg.size >= 1 << 24                             # the sorted / tiled form (max_d <= 2) or the brute-force kernel
    assert sparse == (n_q > 10_000)
    wam, wdist = ops.nearest_bounded(q, tg, max_d)
    for dtype in bd.BARCODE_DTYPES:
        am, dist = bd.nearest_bounded(cuda(q, dtype), cuda(tg, dtype), max_d)
        assert am.dtype == torch.int32 and dist.dtype == torch.uint8
        assert np.array_equal(npy(am), wam) and np.array_equal(npy(dist), wdist)
    sel = rng.choice(q.size, min(q.size, 2500), replace=False)
    oam, odist = orc.nearest(q[sel], tg, max_d)
    assert np.array_equal(wam[sel], oam) and np.array_equal(wdist[sel], odist)
    assert (wam >= 0).sum() > q.size // 4


def test_nearest_ties_and_duplicates_take_the_first_target():
    rng = synth.rng_for(75)
    base = randu32(rng, 50)
    tg = np.concatenate([base ^ np.uint32(3), base, base, base ^ np.uint32(1 << 30)])   # every query has several targets at d = 1
    q = base ^ np.uint32(1 << 10)
    am, dist = (npy(x) for x in bd.nearest_bounded(cuda(q), cuda(tg), 2))
    wam, wdist = ops.nearest_bounded(q, tg, 2)
    oam, odist = orc.nearest(q, tg, 2)
    assert np.array_equal(am, wam) and np.array_equal(dist, wdist) and np.array_equal(am, oam) and np.array_equal(dist, odist)
    assert (dist <= 1).all() and (am < 100).all()


def test_nearest_without_targets():
    q = cuda(np.arange(100, dtype=np.uint32))
    am, dist = bd.nearest_bounded(q, cuda(np.empty(0, np.uint32)), 2)
    assert (npy(am) == -1).all() and (npy(dist) == 255).all()
    am, dist = bd.nearest_bounded(cuda(np.empty(0, np.uint32)), q, 2)
    assert am.numel() == 0 and dist.numel() == 0


# ---------------------------------------------------------------------------------------------------------- a-5 k-mer lookup
@pytest.mark.parametrize("W", [20_000, 3000])
def test_kmer_index_matches_host(W):
    """W >= 4096: posting lists; below: the scan of every string (the index reports which)."""
    rng = synth.rng_for(80 + W % 7)
    wl = whitelist(rng, W)
    wl[:LOW_COMPLEXITY.size] = LOW_COMPLEXITY
    q = near_queries(rng, wl, 1500)
    hix = ops.KmerIndex(wl)
    dix = bd.KmerIndex(cuda(wl, torch.uint32))
    assert dix.info()["postings"] == hix.info()["postings"] == (W >= 4096)
    for mk in (1, 4, 11):
        want = hix.query(q, min_kmers=mk)
        got = dix.query(cuda(q), min_kmers=mk)
        assert got[0].dtype == torch.int32 and got[1].dtype == torch.int32 and got[2].dtype == torch.uint8
        assert got[3].dtype == torch.uint8 and got[3].shape == (want[0].size, 11)
        assert_same_hits(got, want)
        assert want[0].size > (q.size if mk < 11 else 20)
        sample = np.concatenate([rng.choice(q.size - LOW_COMPLEXITY.size, 25, replace=False), q.size - 1 - np.arange(LOW_COMPLEXITY.size)])
        assert_hits_match_oracle(got, q, wl, mk, sample)
    assert dix.info()["kernel_ms"] > 0
    hix.free(); dix.free()


def test_kmer_index_capacity_retry_and_hint():
    rng = synth.rng_for(84)
    wl = whitelist(rng, 10_000)
    q = near_queries(rng, wl, 300)
    want = ops.KmerIndex(wl).query(q, min_kmers=2)
    ix = bd.KmerIndex(cuda(wl))
    assert_same_hits(ix.query(cuda(q), min_kmers=2, cap=1), want)             # BDG_ERR_CAPACITY, then the exact size
    assert ix._room[0] >= want[0].size                                         # the room the call needed, for the next one
    assert_same_hits(ix.query(cuda(q), min_kmers=2), want)                    # the hint is the first guess now
    ix.free()


@pytest.mark.parametrize("n_q", [30, 500])
def test_kmer_score_one_off_matches_host(n_q):
    """Posting lists from 64 queries upwards, the scan below (the rule of bdg_kmer_score)."""
    rng = synth.rng_for(86 + n_q)
    wl = whitelist(rng, 8000)
    wl[:LOW_COMPLEXITY.size] = LOW_COMPLEXITY
    q = near_queries(rng, wl, 500)[-n_q:]
    for mk in (1, 4, 11):
        got = bd.kmer_score(cuda(q), cuda(wl), min_kmers=mk)
        assert_same_hits(got, ops.kmer_score(q, wl, min_kmers=mk))
        assert_hits_match_oracle(got, q, wl, mk, np.arange(0, q.size, max(q.size // 20, 1)))
    assert_same_hits(bd.kmer_score(cuda(q), cuda(wl), min_kmers=3, cap=1), ops.kmer_score(q, wl, min_kmers=3))
    empty = bd.kmer_score(cuda(q), cuda(np.empty(0, np.uint32)))
    assert all(x.shape[0] == 0 for x in empty) and empty[3].shape == (0, 11)
    assert all(x.shape[0] == 0 for x in bd.kmer_score(cuda(np.empty(0, np.uint32)), cuda(wl)))


@pytest.mark.parametrize("W", [20_000, 3000])
def test_kmer_query_guard_bands(W):
    """bdg_dev_kmer_index_query writes nothing outside its caller's buffers of cap hits: sentinel bands around each of them stay
    intact at the exact capacity (where the interior equals the result of bd.KmerIndex.query) and at one less (where the call
    reports BDG_ERR_CAPACITY, d_pos is untouched and only cap entries of the others may be written)."""
    rng = synth.rng_for(88)
    wl = whitelist(rng, W)
    q = near_queries(rng, wl, 400)
    ix = bd.KmerIndex(cuda(wl))
    want = ix.query(cuda(q), min_kmers=3)
    n = want[0].numel()
    assert n > 1000
    G, S = 4096, 0xA5
    L = badger_b200.lib()
    d_q = cuda(q)
    for cap in (n, n - 1):
        bufs = {"hq": torch.full((cap + 2 * G,), -0x5A5A5A5B, dtype=torch.int32, device=bd._device()),
                "hw": torch.full((cap + 2 * G,), -0x5A5A5A5B, dtype=torch.int32, device=bd._device()),
                "cnt": torch.full((cap + 2 * G,), S, dtype=torch.uint8, device=bd._device()),
                "pos": torch.full(((cap + 2 * G) * 11,), S, dtype=torch.uint8, device=bd._device())}
        inner = {k: (v[G * 11:(G + cap) * 11] if k == "pos" else v[G:G + cap]) for k, v in bufs.items()}
        before = {k: v.clone() for k, v in bufs.items()}
        total = C.c_size_t(0)
        rc = L.bdg_dev_kmer_index_query(ix._h, d_q.data_ptr(), q.size, 3, cap, inner["hq"].data_ptr(), inner["hw"].data_ptr(),
                                        inner["cnt"].data_ptr(), inner["pos"].data_ptr(), C.byref(total), bd._stream())
        assert int(total.value) == n
        for k, v in bufs.items():
            lo, hi = (G * 11, (G + cap) * 11) if k == "pos" else (G, G + cap)
            assert torch.equal(v[:lo], before[k][:lo]) and torch.equal(v[hi:], before[k][hi:]), k
        if cap == n:
            assert rc == 0
            assert_same_hits((inner["hq"], inner["hw"], inner["cnt"], inner["pos"].view(cap, 11)), want)
        else:
            assert rc == badger_b200._lib.BDG_ERR_CAPACITY
            assert torch.equal(inner["pos"], before["pos"][G * 11:(G + cap) * 11])
    ix.free()


# ---------------------------------------------------------------------------------------------------------- ordering, traffic
def test_stream_order_without_synchronisation():
    """Inputs come from a kernel queued on a side stream behind a long sleep; the calls run under that stream and nobody
    synchronises: the library must wait for the inputs, and the outputs must be complete when read on that stream."""
    rng = synth.rng_for(91)
    wl = whitelist(rng, 300_000)
    tg = wl[rng.integers(0, wl.size, 3000)]
    q = near_queries(rng, tg, 200_000)                              # members, near a target, and with shared 6-mers
    want_hit = ops.member_sorted(wl, q)
    want_near = ops.nearest_bounded(q[:50_000], tg, 2)
    want_k = ops.KmerIndex(wl).query(q[:2000], min_kmers=4)
    want_s = ops.kmer_score(q[:300], tg, min_kmers=4)
    key = 0x5A5A5A5A
    src_wl, src_q, src_tg = cuda(wl) ^ key, cuda(q) ^ key, cuda(tg) ^ key
    torch.cuda.synchronize()
    side = torch.cuda.Stream(device=bd._device())
    with torch.cuda.stream(side):
        torch.cuda._sleep(200_000_000)
        d_wl, d_q = src_wl ^ key, src_q ^ key
        hit = bd.member_sorted(d_wl, d_q).cpu()
        torch.cuda._sleep(200_000_000)
        d_tg = src_tg ^ key
        near = [x.cpu() for x in bd.nearest_bounded(d_q[:50_000], d_tg, 2)]
        torch.cuda._sleep(200_000_000)
        ix = bd.KmerIndex(src_wl ^ key)
        torch.cuda._sleep(200_000_000)
        k = [x.cpu() for x in ix.query(src_q[:2000] ^ key, min_kmers=4)]
        torch.cuda._sleep(200_000_000)
        s = [x.cpu() for x in bd.kmer_score(src_q[:300] ^ key, src_tg ^ key, min_kmers=4)]
    assert np.array_equal(host(hit), want_hit)
    assert np.array_equal(npy(near[0]), want_near[0]) and np.array_equal(npy(near[1]), want_near[1])
    assert want_hit.sum() > 10_000 and (want_near[0] >= 0).sum() > 10_000 and want_k[0].size > 10_000 and want_s[0].size > 100
    assert_same_hits(k, want_k)
    assert_same_hits(s, want_s)
    ix.free()


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


def test_no_per_query_or_per_hit_array_crosses_pcie(tmp_path):
    from torch.profiler import ProfilerActivity, profile
    rng = synth.rng_for(93)
    wl = whitelist(rng, 1_000_000)
    q = near_queries(rng, wl, 400_000)
    tg = wl[rng.integers(0, wl.size, 10_000)]
    d_wl, d_tg = cuda(wl), cuda(tg)
    ix, hix = bd.KmerIndex(d_wl), ops.KmerIndex(wl)
    moved = {}
    for n in (100_000, 400_000):
        d_q = cuda(q[:n])
        runs = {"device": lambda: (bd.member_sorted(d_wl, d_q), bd.nearest_bounded(d_q[:n // 10], d_tg, 2), ix.query(d_q[:n // 100], min_kmers=4)),
                "host": lambda: (ops.member_sorted(wl, q[:n]), ops.nearest_bounded(q[:n // 10], tg, 2), hix.query(q[:n // 100], min_kmers=4))}
        for form, run in runs.items():
            run()                                                          # warm: the capacity hint of the index is set
            torch.cuda.synchronize()
            out = tmp_path / ("%s_%d" % (form, n))
            out.mkdir()
            with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
                run()
                torch.cuda.synchronize()
            prof.export_chrome_trace(str(out / "trace.json"))
            moved[form, n] = memcpy_bytes(str(out))
    print("PCIe bytes:", moved)
    assert moved["host", 400_000] > 4 * 400_000                            # the count sees the per-query copies of the host forms
    assert moved["device", 400_000] < 4096
    assert moved["device", 400_000] <= moved["device", 100_000] + 64
    ix.free(); hix.free()


# ---------------------------------------------------------------------------------------------------------- errors, contexts
def test_errors_leave_the_library_usable():
    rng = synth.rng_for(95)
    wl = whitelist(rng, 5000)
    q = near_queries(rng, wl, 500)
    d_wl, d_q = cuda(wl), cuda(q)
    want_hit = ops.member_sorted(wl, q)
    want_k = ops.KmerIndex(wl).query(q, min_kmers=4)
    ix = bd.KmerIndex(d_wl)

    def still_works():
        assert np.array_equal(host(bd.member_sorted(d_wl, d_q)), want_hit)
        assert_same_hits(ix.query(d_q, min_kmers=4), want_k)

    bad_args = [
        (ValueError, lambda: bd.member_sorted(torch.from_numpy(wl.view(np.int32)), d_q)),          # CPU tensor
        (ValueError, lambda: bd.member_sorted(d_wl, torch.stack([d_q, d_q], 1)[:, 0])),           # not contiguous
        (TypeError, lambda: bd.member_sorted(d_wl.to(torch.int64), d_q)),                          # wrong dtype
        (ValueError, lambda: bd.nearest_bounded(d_q.view(-1, 1), d_wl)),                          # two dimensions
        (TypeError, lambda: bd.nearest_bounded(d_q, d_wl.float())),
        (badger_b200.BadgerB200Error, lambda: bd.nearest_bounded(d_q, d_wl, 16)),                  # max_d beyond the packed key
        (TypeError, lambda: bd.KmerIndex(d_wl.to(torch.int16))),
        (ValueError, lambda: bd.KmerIndex(d_wl.cpu())),
        (ValueError, lambda: ix.query(d_q.cpu())),
        (TypeError, lambda: ix.query(d_q.to(torch.int64))),
        (TypeError, lambda: bd.kmer_score(d_q, d_wl.to(torch.uint8))),
    ]
    if torch.cuda.device_count() >= 2:
        bad_args.append((ValueError, lambda: ix.query(d_q.to("cuda:1"))))                        # not the first claimed device
    for exc, call in bad_args:
        with pytest.raises(exc):
            call()
        still_works()
    # 2^31 queries or strings: the hit indices are int32
    big = torch.empty(1 << 31, dtype=torch.int32, device=bd._device())
    with pytest.raises(ValueError):
        ix.query(big)
    with pytest.raises(ValueError):
        bd.KmerIndex(big)
    del big
    still_works()
    # the C ABI refuses host memory where it takes device pointers
    L, ERR_ARG = badger_b200.lib(), badger_b200._lib.BDG_ERR_ARG
    h, total = C.c_void_p(), C.c_size_t(0)
    assert L.bdg_dev_kmer_index_create(wl.ctypes.data, wl.size, bd._stream(), C.byref(h)) == ERR_ARG and not h.value
    assert L.bdg_dev_kmer_index_query(ix._h, q.ctypes.data, q.size, 4, 0, None, None, None, None, C.byref(total), bd._stream()) == ERR_ARG
    out = torch.empty(10, dtype=torch.int32, device=bd._device())
    assert L.bdg_dev_kmer_index_query(ix._h, d_q.data_ptr(), q.size, 4, 10, out.data_ptr(), out.data_ptr(), out.data_ptr(),
                                      q.ctypes.data, C.byref(total), bd._stream()) == ERR_ARG
    assert L.bdg_dev_whitelist_check(wl.ctypes.data, wl.size, bd._stream()) == ERR_ARG
    still_works()
    ix.free()
    with pytest.raises(ValueError):
        ix.query(d_q)                                                                          # a freed index


def test_an_index_outlives_a_new_init():
    """An index is built before badger_b200.init claims another set of contexts and queried after it: it stays where it was built,
    and keeps answering while that device is the first claimed one (two contexts on it when the box has one GPU)."""
    rng = synth.rng_for(97)
    wl = whitelist(rng, 30_000)
    q = near_queries(rng, wl, 500)
    want = ops.KmerIndex(wl).query(q, min_kmers=4)
    badger_b200.init([0])
    ix = bd.KmerIndex(cuda(wl))
    assert_same_hits(ix.query(cuda(q), min_kmers=4), want)
    n_dev = torch.cuda.device_count()
    badger_b200.init([0, 0] if n_dev < 2 else [0, 1])
    assert_same_hits(ix.query(cuda(q), min_kmers=4), want)
    if n_dev >= 2:
        badger_b200.init([1, 0])                                        # device 1 is the first claimed device now: refused
        with pytest.raises(badger_b200.BadgerB200Error):
            ix.query(torch.from_numpy(q.view(np.int32)).to("cuda:1"))
        badger_b200.init([0])
        assert_same_hits(ix.query(cuda(q), min_kmers=4), want)
    ix.free()


def test_two_device_contexts_match_one():
    """init([0, 0]) when the box has one GPU (two contexts on the same device), every device otherwise."""
    n_dev = badger_b200.init()
    many = None if n_dev >= 2 else [0, 0]
    rng = synth.rng_for(99)
    wl = whitelist(rng, 200_000)
    tg = wl[rng.integers(0, wl.size, 2000)]
    q = near_queries(rng, tg, 100_000)
    res = []
    for devs in ([0], many):
        badger_b200.init(devs)
        d_wl, d_q, d_tg = cuda(wl), cuda(q), cuda(tg)
        hit = host(bd.member_sorted(d_wl, d_q))
        am, dist = (npy(x) for x in bd.nearest_bounded(d_q, d_tg, 2))
        ix = bd.KmerIndex(d_wl)
        k = canonical_hits(*ix.query(d_q[:3000], min_kmers=4))
        s = canonical_hits(*bd.kmer_score(d_q[:40], d_tg, min_kmers=4))
        ix.free()
        assert np.array_equal(hit, ops.member_sorted(wl, q))
        wam, wdist = ops.nearest_bounded(q, tg, 2)
        assert np.array_equal(am, wam) and np.array_equal(dist, wdist)
        assert_same_hits(k, ops.KmerIndex(wl).query(q[:3000], min_kmers=4))
        assert_same_hits(s, ops.kmer_score(q[:40], tg, min_kmers=4))
        assert hit.sum() > 1000 and (am >= 0).sum() > 1000 and k[0].size > 1000 and s[0].size > 10
        res.append((hit, am, dist, k, s))
    for a, b in zip(res[0], res[1]):
        if isinstance(a, tuple):
            assert all(np.array_equal(x, y) for x, y in zip(a, b))
        else:
            assert np.array_equal(a, b)
