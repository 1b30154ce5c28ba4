"""Per-pair device arithmetic (badger_b200/csrc/bdg_core.cuh), compiled for the host, against the oracle.

The same header is what the CUDA kernels include; this test is the CPU-side proof that the prefilters
are sound (never reject a pair with D <= t) and that the exact stage equals the reference's distances.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from badger_b200 import synth
from oracle import oracle as orc

HERE = os.path.dirname(os.path.abspath(__file__))
u32p = np.ctypeslib.ndpointer(dtype=np.uint32, flags="C_CONTIGUOUS")
u8p = np.ctypeslib.ndpointer(dtype=np.uint8, flags="C_CONTIGUOUS")
u64p = np.ctypeslib.ndpointer(dtype=np.uint64, flags="C_CONTIGUOUS")


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("shim") / "core_host_shim.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-x", "c++",
                           os.path.join(HERE, "core_host_shim.cpp"), "-o", so])
    L = C.CDLL(so)
    L.shim_pairs.argtypes = [u32p, u32p, C.c_size_t] + [u8p] * 8 + [u64p]
    L.shim_edge.argtypes = [C.c_uint32, C.c_uint32, C.c_int]
    L.shim_edge.restype = C.c_int
    L.shim_split.argtypes = [u32p, u32p, C.c_size_t] + [u8p] * 4
    L.shim_pass_pred.argtypes = [C.c_int, u32p, u32p, C.c_size_t, u8p]
    L.shim_pass_possible.argtypes = [C.c_int, C.c_int] + [C.c_uint32] * 4
    L.shim_pass_possible.restype = C.c_int
    L.shim_quick.argtypes = [C.c_int, u32p, u32p, C.c_size_t, u8p]
    L.shim_quick_any.argtypes = [C.c_int, u32p, u32p, C.c_size_t, u8p]
    L.shim_top_possible.argtypes = [C.c_int] + [C.c_uint32] * 4
    L.shim_top_possible.restype = C.c_int
    L.shim_scheme.argtypes = [C.c_void_p, C.c_int]
    L.shim_scheme_first.argtypes = [u32p, u32p, C.c_size_t, u8p, u8p]
    L.shim_scheme_keys.argtypes = [C.c_int, u32p, u32p, C.c_size_t, u32p, u32p, u8p]
    L.shim_join_emulate.argtypes = [u32p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
    L.shim_join_emulate.restype = C.c_size_t
    L.shim_qgram_compact.argtypes = [u32p, u32p, C.c_size_t, u8p, u8p]
    L.shim_kmer_post_emulate.argtypes = [u32p, C.c_size_t, u32p, C.c_size_t, C.c_int, u32p, u32p, u8p, C.c_size_t, u64p]
    L.shim_kmer_post_emulate.restype = C.c_size_t
    return L


def run(shim, a, b):
    n = a.size
    outs = [np.zeros(n, np.uint8) for _ in range(8)]
    mult = np.zeros(n, np.uint64)
    shim.shim_pairs(a, b, n, *outs, mult)
    return dict(zip(["pre1", "pre2", "dsmall", "dplain", "dfull", "da15", "db15", "S"], outs)), mult


def edit_ops(rng, a, k):
    """Apply k random edit operations to the 16-mer a, keep 16 bases (pad randomly)."""
    s = [(a >> (2 * i)) & 3 for i in range(16)]
    for _ in range(k):
        op = rng.integers(0, 3); pos = int(rng.integers(0, len(s)))
        if op == 0:
            s[pos] = (s[pos] + int(rng.integers(1, 4))) & 3
        elif op == 1:
            s.insert(pos, int(rng.integers(0, 4)))
        else:
            del s[pos]
    while len(s) < 16:
        s.append(int(rng.integers(0, 4)))
    return sum(c << (2 * i) for i, c in enumerate(s[:16]))


def make_pairs(seed, n_near=60000, n_rand=20000, n_low=20000):
    rng = np.random.default_rng(seed)
    a, b = [], []
    for _ in range(n_near):
        x = int(rng.integers(0, 1 << 32))
        if rng.random() < 0.3:   # low-complexity seeds exercise the multiplicity side of S
            unit = int(rng.integers(0, 1 << (2 * int(rng.integers(1, 5)))))
            ul = max(1, unit.bit_length() + 1) // 2 or 1
            x = 0
            for i in range(16):
                x |= ((unit >> (2 * (i % ul))) & 3) << (2 * i)
        y = edit_ops(rng, x, int(rng.integers(1, 5)))
        if x != y:
            a.append(x); b.append(y)
    ra = rng.integers(0, 1 << 32, n_rand, dtype=np.uint64); rb = rng.integers(0, 1 << 32, n_rand, dtype=np.uint64)
    a += ra.tolist(); b += rb.tolist()
    # pairs sharing long stretches on shifted diagonals
    for _ in range(n_low):
        x = int(rng.integers(0, 1 << 32)); sh = int(rng.integers(1, 4)) * 2
        y = ((x << sh) | int(rng.integers(0, 1 << sh))) & 0xFFFFFFFF if rng.random() < 0.5 else (x >> sh) | (int(rng.integers(0, 1 << sh)) << (32 - sh))
        if rng.random() < 0.5:
            y = edit_ops(rng, y, 1)
        if x != y:
            a.append(x); b.append(y)
    a = np.asarray(a, dtype=np.uint32); b = np.asarray(b, dtype=np.uint32)
    keep = a != b
    return a[keep], b[keep]


def test_core_vs_oracle(shim):
    a, b = make_pairs(5)
    res, mult = run(shim, a, b)
    L = orc.lib()
    n = a.size
    ed = np.fromiter((L.orc_ed(int(x), 16, int(y), 16) for x, y in zip(a, b)), np.int32, n)
    ea = np.fromiter((L.orc_ed(int(x), 15, int(y), 16) for x, y in zip(a, b)), np.int32, n)
    eb = np.fromiter((L.orc_ed(int(x), 16, int(y), 15) for x, y in zip(a, b)), np.int32, n)
    D = np.minimum(ed, np.minimum(ea, eb))
    S = np.fromiter((L.orc_S(int(x), int(y)) for x, y in zip(a, b)), np.int32, n)
    assert np.array_equal(res["dfull"], ed)
    assert np.array_equal(res["da15"], ea)
    assert np.array_equal(res["db15"], eb)
    assert np.array_equal(res["S"], S)
    assert np.array_equal(res["dsmall"], np.minimum(D, 3))
    assert np.array_equal(res["dplain"], np.minimum(ed, 3))
    # soundness of the prefilters: D<=t  =>  prefilter passes
    assert res["pre1"][D <= 1].all()
    assert res["pre2"][D <= 2].all()
    assert (D <= 1).sum() > 5000 and ((D == 2).sum() > 5000)
    # the prefilters do reject random pairs
    rng = np.random.default_rng(1)
    ra = rng.integers(0, 1 << 32, 1 << 20, dtype=np.uint64).astype(np.uint32)
    rb = rng.integers(0, 1 << 32, 1 << 20, dtype=np.uint64).astype(np.uint32)
    rr, _ = run(shim, ra, rb)
    assert rr["pre1"].mean() < 4e-4      # expected 2*2^-16 + 2*2^-14 = 1.5e-4
    assert rr["pre2"].mean() < 0.012     # expected 9 * 2^-10   = 0.88 %
    # symmetry
    res2, _ = run(shim, b, a)
    for k in ("pre1", "dsmall", "dplain", "S"):   # pre2 is frame-dependent (sound either way)
        assert np.array_equal(res[k], res2[k]), k
    # multiplicities: sum over positions == S, and equal to the oracle's kmer_score multiplicities
    nib = np.stack([(mult >> np.uint64(4 * p)) & np.uint64(15) for p in range(11)], 1).astype(np.int32)
    assert np.array_equal(nib.sum(1), S)
    idx = np.arange(0, n, 97)
    for i in idx:
        _, m = orc.kmer_score(a[i:i + 1], b[i:i + 1])
        assert m[0, 0].tolist() == nib[i].tolist()


def test_edge_predicate_on_golden(shim, gold_pairs):
    for p in gold_pairs["pairs"]:
        for t in range(0, 5):
            want = p["D"] if (p["S"] >= orc.T(t) and p["D"] <= t) else 0
            assert shim.shim_edge(p["ra"], p["rb"], t) == want
            assert shim.shim_edge(p["rb"], p["ra"], t) == want


def test_exhaustive_neighbourhood(shim):
    """Every string within two edit operations of a few seeds (incl. truncation effects)."""
    rng = np.random.default_rng(9)
    seeds = [int(rng.integers(0, 1 << 32)) for _ in range(3)] + [0, 0x11111111 * 0 + 0x44444444, int(synth.rank_many(["ACACACACACACACAC"])[0])]
    for x in seeds:
        s = [(x >> (2 * i)) & 3 for i in range(16)]
        neigh = set()

        def one(seq):
            out = []
            for pos in range(len(seq)):
                for c in range(4):
                    if c != seq[pos]:
                        out.append(seq[:pos] + [c] + seq[pos + 1:])
                out.append(seq[:pos] + seq[pos + 1:])
            for pos in range(len(seq) + 1):
                for c in range(4):
                    out.append(seq[:pos] + [c] + seq[pos:])
            return out

        lvl1 = one(s)
        sample = [lvl1[i] for i in rng.choice(len(lvl1), 40, replace=False)]
        lvl2 = [y for z in sample for y in one(z)]
        for seq in lvl1 + lvl2:
            for pad in range(4):
                q = (seq + [pad, pad])[:16] if len(seq) < 16 else seq[:16]
                neigh.add(sum(c << (2 * i) for i, c in enumerate(q)))
        neigh.discard(x)
        b = np.fromiter(neigh, dtype=np.uint32)
        a = np.full(b.size, x, dtype=np.uint32)
        res, _ = run(shim, a, b)
        L = orc.lib()
        D = np.fromiter((L.orc_D(int(x), int(y)) for y in b), np.int32, b.size)
        assert np.array_equal(res["dsmall"], np.minimum(D, 3))
        assert res["pre1"][D <= 1].all() and res["pre2"][D <= 2].all()


def split(shim, a, b):
    outs = [np.zeros(a.size, np.uint8) for _ in range(4)]
    shim.shim_split(a, b, a.size, *outs)
    return dict(zip(["l1", "t1", "l2", "t2"], outs))


def test_split_filters_sound(shim):
    """light || top is a necessary condition for D <= t in both frames (bdg_core.cuh, tiled edge kernel)."""
    L = orc.lib()
    tot1 = tot2 = 0
    for seed in (5, 6, 7):
        a, b = make_pairs(seed)
        D = np.fromiter((L.orc_D(int(x), int(y)) for x, y in zip(a, b)), np.int32, a.size)
        for x, y in ((a, b), (b, a)):
            r = split(shim, x, y)
            assert (r["l1"] | r["t1"])[D <= 1].all()
            assert (r["l2"] | r["t2"])[D <= 2].all()
        tot1 += int((D <= 1).sum()); tot2 += int((D == 2).sum())
    assert tot1 > 15000 and tot2 > 15000
    rng = np.random.default_rng(2)
    ra = rng.integers(0, 1 << 32, 1 << 20, dtype=np.uint64).astype(np.uint32)
    rb = rng.integers(0, 1 << 32, 1 << 20, dtype=np.uint64).astype(np.uint32)
    r = split(shim, ra, rb)
    assert r["l1"].mean() < 6e-5 and r["t1"].mean() < 3e-4         # 2^-15 ; 2^-16 + 2*2^-14
    assert r["l2"].mean() < 6e-3 and r["t2"].mean() < 4.5e-3       # 4*2^-10 ; 3*2^-10


def test_split_filters_exhaustive_neighbourhood(shim):
    """All strings within two operations of a few seeds, all paddings: no edge candidate is lost."""
    rng = np.random.default_rng(11)
    L = orc.lib()
    seeds = [int(rng.integers(0, 1 << 32)) for _ in range(4)] + [0, 0xFFFFFFFF, 0x44444444, int(synth.rank_many(["ACACACACACACACAC"])[0])]
    for x in seeds:
        s = [(x >> (2 * i)) & 3 for i in range(16)]

        def one(seq):
            out = []
            for pos in range(len(seq)):
                for c in range(4):
                    if c != seq[pos]:
                        out.append(seq[:pos] + [c] + seq[pos + 1:])
                out.append(seq[:pos] + seq[pos + 1:])
            for pos in range(len(seq) + 1):
                for c in range(4):
                    out.append(seq[:pos] + [c] + seq[pos:])
            return out

        lvl1 = one(s)
        sample = [lvl1[i] for i in rng.choice(len(lvl1), 60, replace=False)]
        neigh = set()
        for seq in lvl1 + [y for z in sample for y in one(z)]:
            for pad in range(16):
                q = (seq + [pad & 3, pad >> 2])[:16]
                neigh.add(sum(c << (2 * i) for i, c in enumerate(q)))
        neigh.discard(x)
        b = np.fromiter(neigh, dtype=np.uint32)
        a = np.full(b.size, x, dtype=np.uint32)
        D = np.fromiter((L.orc_D(int(x), int(y)) for y in b), np.int32, b.size)
        for p, q in ((a, b), (b, a)):
            r = split(shim, p, q)
            assert (r["l1"] | r["t1"])[D <= 1].all()
            assert (r["l2"] | r["t2"])[D <= 2].all()


@pytest.mark.parametrize("t", [1, 2])
def test_top_possible_is_conservative(shim, t):
    """If some pair of a (row run) x (column run) tile of a sorted array meets a top condition, the interval test
    on the runs' end points must say so."""
    rng = np.random.default_rng(20 + t)
    checked = hits = skipped = 0
    for n, rows, cols in ((3000, 64, 32), (20000, 256, 128), (200000, 256, 256)):
        base = rng.integers(0, 1 << 32, n, dtype=np.uint64).astype(np.uint32)
        # plant near-duplicates so that top conditions do occur
        extra = (base[: n // 4] ^ rng.integers(0, 1 << 12, n // 4, dtype=np.uint64).astype(np.uint32))
        s = np.unique(np.concatenate([base, extra]))
        for _ in range(300):
            r0 = int(rng.integers(0, s.size - rows)); c0 = int(rng.integers(0, s.size - cols))
            if rng.random() < 0.3:
                c0 = min(s.size - cols, r0 + int(rng.integers(0, rows)))
            A = s[r0:r0 + rows]; B = s[c0:c0 + cols]
            aa = np.repeat(A, B.size); bb = np.tile(B, A.size)
            r = split(shim, aa, bb)
            any_top = bool(r["t%d" % t].any())
            poss = bool(shim.shim_top_possible(t, int(A[0]), int(A[-1]), int(B[0]), int(B[-1])))
            assert poss or not any_top
            checked += 1; hits += any_top; skipped += (not poss)
    assert hits > 50 and skipped > 200


def pass_mask(shim, t, a, b):
    m = np.zeros(a.size, np.uint8)
    shim.shim_pass_pred(t, a, b, a.size, m)
    assert not (m & 0x80).any(), "pass_pred and pass_pred_rot disagree"
    return m


def rotl(v, r):
    v = v.astype(np.uint32)
    return v if r == 0 else ((v << np.uint32(r)) | (v >> np.uint32(32 - r))).astype(np.uint32)


PASS_ROT = {1: [0, 16], 2: [0, 10, 20]}


@pytest.mark.parametrize("t", [1, 2])
def test_pass_predicates_cover_and_are_symmetric(shim, t):
    """Sparse edge passes: every pair with D <= t fires in at least one pass; predicates are orientation-free."""
    L = orc.lib()
    tot = 0
    for seed in (5, 8):
        a, b = make_pairs(seed)
        D = np.fromiter((L.orc_D(int(x), int(y)) for x, y in zip(a, b)), np.int32, a.size)
        m = pass_mask(shim, t, a, b)
        assert np.array_equal(m, pass_mask(shim, t, b, a))
        assert (m[D <= t] != 0).all()
        tot += int((D <= t).sum())
    assert tot > 10000
    rng = np.random.default_rng(3)
    ra = rng.integers(0, 1 << 32, 1 << 20, dtype=np.uint64).astype(np.uint32)
    rb = rng.integers(0, 1 << 32, 1 << 20, dtype=np.uint64).astype(np.uint32)
    assert (pass_mask(shim, t, ra, rb) != 0).mean() < (4e-4 if t == 1 else 0.014)


@pytest.mark.parametrize("t", [1, 2])
def test_pass_possible_is_conservative(shim, t):
    """Interval test of every pass on arrays sorted by that pass's rotated key."""
    rng = np.random.default_rng(40 + t)
    for p, rot in enumerate(PASS_ROT[t]):
        hits = skipped = 0
        for n, rows, cols in ((3000, 64, 32), (20000, 256, 128), (200000, 256, 128)):
            base = rng.integers(0, 1 << 32, n, dtype=np.uint64).astype(np.uint32)
            noise = rng.integers(0, 1 << 12, n // 4, dtype=np.uint64).astype(np.uint32)
            extra = base[: n // 4] ^ rotl(noise, int(rng.integers(0, 32)))
            s = np.unique(rotl(np.concatenate([base, extra]), rot))       # sorted by the rotated key
            for _ in range(250):
                r0 = int(rng.integers(0, s.size - rows)); c0 = int(rng.integers(0, s.size - cols))
                if rng.random() < 0.3:
                    c0 = min(s.size - cols, r0 + int(rng.integers(0, rows)))
                A = s[r0:r0 + rows]; B = s[c0:c0 + cols]
                aa = np.repeat(A, B.size); bb = np.tile(B, A.size)
                fires = ((pass_mask(shim, t, rotl(aa, (32 - rot) % 32), rotl(bb, (32 - rot) % 32)) >> p) & 1).any()
                poss = bool(shim.shim_pass_possible(t, p, int(A[0]), int(A[-1]), int(B[0]), int(B[-1])))
                assert poss or not fires, (t, p)
                hits += bool(fires); skipped += (not poss)
        assert hits > 30 and skipped > 150, (t, p, hits, skipped)


@pytest.mark.parametrize("t", [1, 2])
def test_quick_pass_sound(shim, t):
    """The per-pair test of the sparse passes never rejects a pair with D <= t (both frames), and rejects most others."""
    L = orc.lib()
    for seed in (5, 12):
        a, b = make_pairs(seed)
        D = np.fromiter((L.orc_D(int(x), int(y)) for x, y in zip(a, b)), np.int32, a.size)
        for x, y in ((a, b), (b, a)):
            out = np.zeros(x.size, np.uint8)
            shim.shim_quick(t, x, y, x.size, out)
            assert out[D <= t].all()
    rng = np.random.default_rng(4)
    ra = rng.integers(0, 1 << 32, 1 << 20, dtype=np.uint64).astype(np.uint32)
    rb = rng.integers(0, 1 << 32, 1 << 20, dtype=np.uint64).astype(np.uint32)
    out = np.zeros(ra.size, np.uint8)
    shim.shim_quick(t, ra, rb, ra.size, out)
    assert out.mean() < (0.004 if t == 1 else 0.03)


@pytest.mark.parametrize("t", [2, 3, 5])
def test_quick_pass_any_sound(shim, t):
    """Generic quick test of the dense kernel (t >= 3): never rejects a pair with D <= t, in both frames."""
    L = orc.lib()
    a, b = make_pairs(30 + t, n_near=25000, n_rand=3000, n_low=8000)
    rng = np.random.default_rng(t)
    extra_a, extra_b = [], []
    for _ in range(12000):                      # more operations than make_pairs uses, so that D = 3..5 is well covered
        x = int(rng.integers(0, 1 << 32)); y = edit_ops(rng, x, int(rng.integers(3, 7)))
        if x != y:
            extra_a.append(x); extra_b.append(y)
    a = np.concatenate([a, np.asarray(extra_a, np.uint32)]); b = np.concatenate([b, np.asarray(extra_b, np.uint32)])
    D = np.fromiter((L.orc_D(int(x), int(y)) for x, y in zip(a, b)), np.int32, a.size)
    for x, y in ((a, b), (b, a)):
        out = np.zeros(x.size, np.uint8)
        shim.shim_quick_any(t, x, y, x.size, out)
        assert out[D <= t].all()
    assert (D == t).sum() > 1000
    ra = rng.integers(0, 1 << 32, 1 << 18, dtype=np.uint64).astype(np.uint32)
    rb = rng.integers(0, 1 << 32, 1 << 18, dtype=np.uint64).astype(np.uint32)
    out = np.zeros(ra.size, np.uint8)
    shim.shim_quick_any(t, ra, rb, ra.size, out)
    print("t", t, "random pass rate", out.mean())


# ------------------------------------------------------------------------------------------ two-block seeds (t = 2)
def two_op_neighbourhood(x):
    """Every 16-mer reachable from x by at most two edit operations (all paddings of the shortened ones)."""
    def one(seq):
        out = []
        for pos in range(len(seq)):
            for c in range(4):
                if c != seq[pos]:
                    out.append(seq[:pos] + [c] + seq[pos + 1:])
            out.append(seq[:pos] + seq[pos + 1:])
        for pos in range(len(seq) + 1):
            for c in range(4):
                out.append(seq[:pos] + [c] + seq[pos:])
        return out

    s = [(x >> (2 * i)) & 3 for i in range(16)]
    lvl1 = one(s)
    neigh = set()
    for seq in lvl1 + [y for z in lvl1 for y in one(z)]:
        if len(seq) >= 16:
            neigh.add(sum(c << (2 * i) for i, c in enumerate(seq[:16])))
        else:
            for p1 in range(4):
                for p2 in range(4):
                    neigh.add(sum(c << (2 * i) for i, c in enumerate((seq + [p1, p2])[:16])))
    neigh.discard(x)
    return np.fromiter(neigh, dtype=np.uint32)


SCHEMES = {"4": [4, 4, 4, 3], "5": [3, 3, 3, 3, 3], "6": [3, 3, 3, 2, 2, 2]}


def set_scheme(shim, name):
    bases = SCHEMES[name]
    n = shim.shim_scheme((C.c_int * len(bases))(*bases), len(bases))
    assert n > 0
    return n


def scheme_first(shim, a, b):
    """First (condition, orientation) a pair meets: by the definition and through the flag table; they must agree."""
    slow = np.zeros(a.size, np.uint8); fast = np.zeros(a.size, np.uint8)
    shim.shim_scheme_first(np.ascontiguousarray(a), np.ascontiguousarray(b), a.size, slow, fast)
    assert np.array_equal(slow, fast)
    return slow


def test_seed_scheme_tables(shim):
    """bdg_seed.cuh: number of conditions per block layout, symmetric ones first in every block set, keys of both sides."""
    assert set_scheme(shim, "4") == 13 and shim.shim_scheme_nself() == 6
    assert set_scheme(shim, "5") == 25 and shim.shim_scheme_nself() == 10
    assert set_scheme(shim, "6") == 41 and shim.shim_scheme_nself() == 15
    assert shim.shim_scheme((C.c_int * 3)(5, 5, 4), 3) == -1              # not 15 bases
    rng = np.random.default_rng(4)
    n = 1 << 18
    a = rng.integers(0, 1 << 32, n, dtype=np.uint64).astype(np.uint32)
    b = a ^ (rng.integers(0, 1 << 32, n, dtype=np.uint64).astype(np.uint32) & rng.integers(0, 1 << 32, n, dtype=np.uint64).astype(np.uint32)
             & rng.integers(0, 1 << 32, n, dtype=np.uint64).astype(np.uint32))      # ~1/8 of the bits differ: many key hits, many misses
    for name in SCHEMES:
        nc = set_scheme(shim, name)
        ka = np.zeros(n, np.uint32); kb = np.zeros(n, np.uint32); pred = np.zeros(n, np.uint8)
        fired = np.zeros(n, bool)
        first = scheme_first(shim, np.minimum(a, b), np.maximum(a, b))
        for c in range(nc):
            shim.shim_scheme_keys(c, np.minimum(a, b), np.maximum(a, b), n, ka, kb, pred)
            bits = shim.shim_scheme_key_bits(c)
            assert int(ka.max()) < (1 << bits) and int(kb.max()) < (1 << bits)
            assert np.array_equal(pred.astype(bool), ka == kb)
            assert shim.shim_scheme_row_sort(c) <= c
            fired |= pred.astype(bool) & (first == 2 * c)
        assert fired.sum() > 1000
        # the block sets as the driver walks them: consecutive runs of conditions that share their row order
        set_first = [shim.shim_scheme_set_first(k) for k in range(shim.shim_scheme_nsets() + 1)]
        assert set_first[0] == 0 and set_first[-1] == nc and all(x < y for x, y in zip(set_first, set_first[1:]))
        for k in range(len(set_first) - 1):
            assert all(shim.shim_scheme_row_sort(c) == set_first[k] for c in range(set_first[k], set_first[k + 1]))


@pytest.mark.parametrize("name", ["4", "5", "6"])
def test_seed_conditions_are_necessary_for_d2(shim, name):
    """D(a,b) <= 2 implies that some condition holds for (min, max) or for (max, min): checked on random near pairs,
    low-complexity and shifted pairs, and on the complete two-operation neighbourhoods of random and repetitive seeds."""
    L = orc.lib()
    set_scheme(shim, name)
    tot = 0
    for seed in (5, 8):
        a, b = make_pairs(seed)
        D = np.fromiter((L.orc_D(int(x), int(y)) for x, y in zip(a, b)), np.int32, a.size)
        near = D <= 2
        assert (scheme_first(shim, np.minimum(a, b), np.maximum(a, b))[near] != 255).all()
        tot += int(near.sum())
    assert tot > 50000
    rng = np.random.default_rng(9)
    seeds = [int(rng.integers(0, 1 << 32)) for _ in range(3)] + [0, 0x44444444] + \
        [int(v) for v in synth.rank_many(["ACACACACACACACAC", "AAAAAAAACCCCCCCC", "ACGACGACGACGACGA", "TTTTGTTTTGTTTTGT"])]
    for x in seeds:
        b = two_op_neighbourhood(x)
        a = np.full(b.size, x, dtype=np.uint32)
        D = np.fromiter((L.orc_D(x, int(y)) for y in b), np.int32, b.size)
        near = D <= 2
        assert near.sum() > 1000
        assert (scheme_first(shim, np.minimum(a, b), np.maximum(a, b))[near] != 255).all()
    # and the seeds do select: a random pair meets a condition far less often than a single 5-base block (11 / 1024)
    ra = rng.integers(0, 1 << 32, 1 << 20, dtype=np.uint64).astype(np.uint32)
    rb = rng.integers(0, 1 << 32, 1 << 20, dtype=np.uint64).astype(np.uint32)
    rate = (scheme_first(shim, np.minimum(ra, rb), np.maximum(ra, rb)) != 255).mean()
    assert rate < {"4": 1.3e-3, "5": 2.5e-4, "6": 1.2e-4}[name]


@pytest.mark.parametrize("name", ["4", "5"])
def test_join_passes_reproduce_the_oracle_edge_set(shim, name):
    """The passes of bdg_join.cuh emulated on the host with the kernel's own per-pair functions (sort by key, pair equal-key
    buckets, quick test, dist_small, hand-over table, score): the union over the conditions must be the oracle's edge set at
    t = 2, every edge exactly once."""
    nc = set_scheme(shim, name)
    rng = synth.rng_for(91)
    cells = rng.integers(0, 1 << 32, 120, dtype=np.uint64).astype(np.uint32)
    obs, _ = synth.simulate_reads(cells, 9000, 0.06, rng)
    s = np.unique(obs)
    n = s.size
    wa, wb, wd, _ = orc.Index(s).edges(2)
    cap = 64 * n
    a = np.empty(cap, np.uint32); b = np.empty(cap, np.uint32); d = np.empty(cap, np.uint8)
    st = np.zeros(5 * (nc + 1), np.uint64)
    k = shim.shim_join_emulate(s, n, a.ctypes.data, b.ctypes.data, d.ctypes.data, cap, st.ctypes.data)
    assert k == wa.size and k > 5000
    o = np.lexsort((b[:k], a[:k]))
    assert np.array_equal(a[:k][o], wa) and np.array_equal(b[:k][o], wb) and np.array_equal(d[:k][o], wd)
    tested, passed, near, mine, edges = (int(x) for x in st[:5])
    assert edges == k and mine >= edges and near >= mine and passed >= near and tested >= passed
    assert tested < 0.03 * n * (n - 1) / 2                  # the seeds leave a small share of the pairs (clustered data)


def test_compact_score_equals_the_unrolled_one(shim):
    a, b = make_pairs(11, n_near=30000, n_rand=10000, n_low=20000)
    full = np.zeros(a.size, np.uint8); compact = np.zeros(a.size, np.uint8)
    shim.shim_qgram_compact(a, b, a.size, full, compact)
    assert np.array_equal(full, compact) and full.max() > 50


@pytest.mark.parametrize("min_kmers", [1, 3, 5])
def test_posting_list_form_emits_every_hit_once(shim, min_kmers):
    """a-5 through the 6-mer posting lists (kmer_post_kernel's rule, on the host): the hits, each exactly once, are the oracle's
    (q, w) pairs with S >= min_kmers, found with a few per cent of the Q x W evaluations."""
    rng = np.random.default_rng(41)
    wl = rng.integers(0, 1 << 32, 20000, dtype=np.uint64).astype(np.uint32)
    wl[:20] = np.asarray([0, 0x55555555, 0xAAAAAAAA, 0xFFFFFFFF, 0x11111111, 0x44444444, 0x1B1B1B1B, 0xE4E4E4E4, 0x00000001, 0x40000000] * 2,
                         np.uint32)
    near = wl[rng.integers(0, wl.size, 60)] ^ (np.uint32(3) << (2 * rng.integers(0, 16, 60)).astype(np.uint32))
    q = np.concatenate([wl[:30], near, rng.integers(0, 1 << 32, 60, dtype=np.uint64).astype(np.uint32)])
    cap = 1 << 20
    hq = np.zeros(cap, np.uint32); hw = np.zeros(cap, np.uint32); cnt = np.zeros(cap, np.uint8); ev = np.zeros(1, np.uint64)
    n = shim.shim_kmer_post_emulate(q, q.size, wl, wl.size, min_kmers, hq, hw, cnt, cap, ev)
    assert 0 < n <= cap
    wc, _ = orc.kmer_score(q, wl, want_mult=False)
    wq, ww = np.nonzero(wc >= min_kmers)
    o = np.lexsort((hw[:n], hq[:n]))
    assert np.array_equal(hq[:n][o], wq) and np.array_equal(hw[:n][o], ww) and np.array_equal(cnt[:n][o], wc[wq, ww])
    assert int(ev[0]) < 0.05 * q.size * wl.size
