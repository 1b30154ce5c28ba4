"""The t = 2 join's one-sided quick test and the hand-over that knows the sides (bdg_seed.cuh), compiled for the host.

A shifted condition tests its pairs on the row's diagonal side {0, +1} only, a symmetric one on either side; the hand-over
table is indexed by the block-match flags and two side bits computed by the kernel's own filter function.  Checked here for
the block layouts of 4, 5 and 6 blocks: the table against its definition, every pair with D <= 2 against the rule "has an
owner, and the owner's pass lets it through", and the emulated passes against the oracle's edge set.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from badger_b200 import synth
from oracle import oracle as orc
from test_core_host import SCHEMES, make_pairs, two_op_neighbourhood

HERE = os.path.dirname(os.path.abspath(__file__))
u32p = np.ctypeslib.ndpointer(dtype=np.uint32, flags="C_CONTIGUOUS")
u8p = np.ctypeslib.ndpointer(dtype=np.uint8, flags="C_CONTIGUOUS")
NONE = 255


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("sides") / "join_sides_host_shim.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-x", "c++",
                           os.path.join(HERE, "join_sides_host_shim.cpp"), "-o", so])
    L = C.CDLL(so)
    L.shim_scheme.argtypes = [C.c_void_p, C.c_int]
    L.shim_cond.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    L.shim_tables.argtypes = [u8p, u8p]
    L.shim_owner.argtypes = [u32p, u32p, C.c_size_t, u8p, u8p, u8p, u8p]
    L.shim_filter.argtypes = [C.c_int, u32p, u32p, C.c_size_t, u8p]
    L.shim_join_emulate.argtypes = [u32p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
    L.shim_join_emulate.restype = C.c_size_t
    return L


def set_scheme(shim, name):
    bases = SCHEMES[name]
    n = shim.shim_scheme((C.c_int * len(bases))(*bases), len(bases))
    assert n > 0
    return n


def conditions(shim, nc):
    out = []
    for c in range(nc):
        nf = C.c_int(); blk = (C.c_int * 8)(); d = (C.c_int * 8)()
        self_ = shim.shim_cond(c, C.byref(nf), blk, d)
        out.append((bool(self_), [(blk[k], d[k]) for k in range(nf.value)]))
    return out


def owners(shim, a, b):
    a = np.ascontiguousarray(np.minimum(a, b)); b2 = np.ascontiguousarray(np.maximum(a, b))
    n = a.size
    slow, fast, sides, passes = (np.zeros(n, np.uint8) for _ in range(4))
    shim.shim_owner(a, b2, n, slow, fast, sides, passes)
    return slow, fast, sides, passes


@pytest.mark.parametrize("name", ["4", "5", "6"])
def test_side_table_equals_its_definition(shim, name):
    """Every entry of the side-aware table, recomputed from the condition list: the first (condition, orientation) whose
    block flags are all set and whose filter passes under the index's side bits (symmetric: always; shifted: bit o)."""
    nc = set_scheme(shim, name)
    nflags = shim.shim_nflags()
    lut = np.zeros(1 << nflags, np.uint8); lut_sides = np.zeros(1 << (nflags + 2), np.uint8)
    shim.shim_tables(lut, lut_sides)
    idx = np.arange(1 << (nflags + 2), dtype=np.uint32)
    f, sd = idx & np.uint32((1 << nflags) - 1), idx >> np.uint32(nflags)
    want = np.full(idx.size, NONE, np.uint8)
    for c, (self_, fields) in enumerate(conditions(shim, nc)):
        for o in range(1 if self_ else 2):
            bits = sum(1 << (3 * blk + (0 if d == 0 else 1 + o)) for blk, d in fields)
            hit = ((f & np.uint32(bits)) == bits) & (want == NONE)
            if not self_:
                hit &= ((sd >> np.uint32(o)) & 1) == 1
            want[hit] = 2 * c + o
    assert np.array_equal(lut_sides, want)
    # with both side bits set the rule is the one of the flag table
    assert np.array_equal(lut_sides[3 << nflags:], lut)


@pytest.mark.parametrize("name", ["4", "5", "6"])
def test_every_close_pair_has_an_owner_that_emits_it(shim, name):
    """Random near pairs, low-complexity and shifted pairs, and the complete two-operation neighbourhoods of random and
    repetitive seeds: every pair with D <= 2 has an owner; the table lookup at the index join_process computes names it; the
    owner's key matches and the owner's one-sided (shifted) or either-side (symmetric, both bucket orders) test passes."""
    L = orc.lib()
    set_scheme(shim, name)
    sets = []
    for seed in (5, 8):
        a, b = make_pairs(seed)
        sets.append((a, b))
    rng = np.random.default_rng(9)
    seeds = [int(rng.integers(0, 1 << 32)) for _ in range(2)] + [0, 0x44444444] + \
        [int(v) for v in synth.rank_many(["ACACACACACACACAC", "AAAAAAAACCCCCCCC", "ACGACGACGACGACGA", "TTTTGTTTTGTTTTGT"])]
    for x in seeds:
        b = two_op_neighbourhood(x)
        sets.append((np.full(b.size, x, dtype=np.uint32), b))
    tot = one_sided = 0
    for a, b in sets:
        D = np.fromiter((L.orc_D(int(x), int(y)) for x, y in zip(a, b)), np.int32, a.size)
        slow, fast, sides, passes = owners(shim, a, b)
        assert np.array_equal(slow, fast)
        near = D <= 2
        assert (slow[near] != NONE).all()
        assert (passes[near] == 3).all()
        tot += int(near.sum()); one_sided += int((near & (sides != 3)).sum())
    assert tot > 100000
    assert one_sided > 1000          # pairs that only one orientation's test passes do occur


def test_side_bits_are_the_kernel_filter(shim):
    """seed_side_bits is join2_quick<true> in the two orientations; the symmetric filter is the OR of the two sides, and both
    are at most as permissive as the three-diagonal quick test they replace."""
    rng = np.random.default_rng(17)
    a, b = make_pairs(21, n_near=20000, n_rand=20000, n_low=20000)
    n = a.size
    ab = np.ascontiguousarray(np.minimum(a, b)); ba = np.ascontiguousarray(np.maximum(a, b))
    set_scheme(shim, "5")
    _, _, sides, _ = owners(shim, ab, ba)
    fwd = np.zeros(n, np.uint8); rev = np.zeros(n, np.uint8); sym = np.zeros(n, np.uint8)
    shim.shim_filter(1, ab, ba, n, fwd)
    shim.shim_filter(1, ba, ab, n, rev)
    shim.shim_filter(0, ab, ba, n, sym)
    assert np.array_equal(sides & 1, fwd & 1) and np.array_equal(sides >> 1, rev & 1)
    assert not ((fwd & 1) & ~(fwd >> 1) & 1).any() and not ((sym & 1) & ~(sym >> 1) & 1).any()
    x = rng.integers(0, 1 << 32, 1 << 18, dtype=np.uint64).astype(np.uint32)
    y = np.ascontiguousarray(x ^ (rng.integers(0, 1 << 32, x.size, dtype=np.uint64).astype(np.uint32)
                                  & rng.integers(0, 1 << 32, x.size, dtype=np.uint64).astype(np.uint32)))
    s0 = np.zeros(x.size, np.uint8); s1 = np.zeros(x.size, np.uint8)
    shim.shim_filter(0, x, y, x.size, s0)
    shim.shim_filter(0, y, x, x.size, s1)
    m = lambda v: v.astype(np.uint64) | (v.astype(np.uint64) << np.uint64(1))   # noqa: E731
    for p, q, got in ((x, y, s0), (y, x, s1)):
        def le2(w):
            w = w & np.uint64(0x2AAAAAAA)
            w &= w - np.uint64(1); w &= w - np.uint64(1)
            return w == 0
        pp = le2(m(p ^ q) & m(p ^ (q >> np.uint32(2))))
        pm = le2(m(p ^ q) & m(p ^ ((q << np.uint32(2)) & np.uint32(0xFFFFFFFF))))
        assert np.array_equal(got & 1, (pp | pm).astype(np.uint8))


def low_complexity_set(rng, n):
    units = ["AC", "AAC", "ACGT", "AAAAC", "TTG", "CAG", "ACACG"]
    out = set()
    while len(out) < n:
        u = units[int(rng.integers(0, len(units)))]
        off = int(rng.integers(0, len(u)))
        base = (u * 20)[off:off + 16]
        s = [("ACGT".index(ch)) for ch in base]
        x = sum(c << (2 * i) for i, c in enumerate(s))
        for _ in range(int(rng.integers(0, 4))):
            x ^= int(rng.integers(1, 4)) << (2 * int(rng.integers(0, 16)))
        out.add(x & 0xFFFFFFFF)
    return np.asarray(sorted(out), np.uint32)


@pytest.mark.parametrize("name,kind", [("4", "reads"), ("5", "reads"), ("6", "reads"), ("5", "low"), ("6", "low")])
def test_join_passes_with_sides_reproduce_the_oracle_edge_set(shim, name, kind):
    """The join passes emulated with the one-sided filter and the side-aware table, the buckets in a shuffled order: the union
    over the conditions is the oracle's edge set at t = 2, every edge exactly once, from fewer candidates than the
    three-diagonal quick test lets through."""
    nc = set_scheme(shim, name)
    rng = synth.rng_for(93)
    if kind == "reads":
        cells = rng.integers(0, 1 << 32, 400, dtype=np.uint64).astype(np.uint32)
        obs, _ = synth.simulate_reads(cells, 40000, 0.06, rng)
        s = np.unique(obs)
    else:
        s = low_complexity_set(rng, 20000)
    n = s.size
    assert 20000 <= n <= 50000
    wa, wb, wd, _ = orc.Index(s).edges(2)
    shuffled = np.ascontiguousarray(s[rng.permutation(n)])
    cap = 64 * n
    a = np.empty(cap, np.uint32); b = np.empty(cap, np.uint32); d = np.empty(cap, np.uint8)
    st = np.zeros(6, np.uint64)
    k = shim.shim_join_emulate(shuffled, n, a.ctypes.data, b.ctypes.data, d.ctypes.data, cap, st.ctypes.data)
    assert k == wa.size and k > 2000
    o = np.lexsort((b[:k], a[:k]))
    assert np.array_equal(a[:k][o], wa) and np.array_equal(b[:k][o], wb) and np.array_equal(d[:k][o], wd)
    tested, cand, near, mine, edges, cand_old = (int(x) for x in st)
    assert edges == k and mine >= edges and near >= mine and cand >= near and tested >= cand
    assert cand < cand_old
    print(name, kind, "n", n, "edges", k, "pairs", tested, "candidates", cand, "three-diagonal candidates", cand_old, "nconds", nc)
