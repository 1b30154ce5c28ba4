"""The t = 3 seed scheme of the join form (badger_b200/csrc/bdg_seed3.cuh), compiled for the host, against the oracle.

Necessity (every pair with D <= 3 meets some condition in some orientation), the kernel's hand-over walk against the
definition, and the join passes emulated with the kernel's own per-pair functions against the oracle's edge set."""
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
i32p = np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")
NONE = 0xFFFF
LAYOUTS = {5: [3, 3, 3, 3, 3], 6: [3, 3, 3, 2, 2, 2], 7: [3, 2, 2, 2, 2, 2, 2]}


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("shim3") / "seed3_host_shim.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-x", "c++",
                           os.path.join(HERE, "seed3_host_shim.cpp"), "-o", so])
    L = C.CDLL(so)
    L.shim3_scheme.argtypes = [C.c_void_p, C.c_int]
    L.shim3_first.argtypes = [u32p, u32p, C.c_size_t, i32p, i32p]
    L.shim3_hits.argtypes = [u32p, u32p, C.c_size_t, i32p]
    L.shim3_quick.argtypes = [u32p, u32p, C.c_size_t, u8p]
    L.shim3_neighbourhood.argtypes = [C.c_uint32, C.c_int, C.c_void_p]
    L.shim3_join_emulate.argtypes = [u32p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
    L.shim3_join_emulate.restype = C.c_size_t
    return L


def use_layout(shim, nb):
    bases = (C.c_int * nb)(*LAYOUTS[nb])
    n = shim.shim3_scheme(bases, nb)
    assert n > 0
    return n


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


def periodic(rng):
    unit = int(rng.integers(0, 1 << (2 * int(rng.integers(1, 5)))))
    ul = int(rng.integers(1, 5))
    return sum(((unit >> (2 * (i % ul))) & 3) << (2 * i) for i in range(16))


def near_pairs(seed, n_near=30000, n_shift=8000, n_rand=5000):
    """Random and low-complexity 16-mers with 1-4 random edits, pairs on shifted diagonals, random pairs."""
    rng = np.random.default_rng(seed)
    a, b = [], []
    for _ in range(n_near):
        x = periodic(rng) if rng.random() < 0.3 else int(rng.integers(0, 1 << 32))
        a.append(x); b.append(edit_ops(rng, x, int(rng.integers(1, 5))))
    for _ in range(n_shift):
        x = int(rng.integers(0, 1 << 32)); sh = int(rng.integers(1, 4)) * 2
        y = ((x << sh) | int(rng.integers(0, 1 << sh))) & 0xFFFFFFFF if rng.random() < 0.5 else (x >> sh) | (int(rng.integers(0, 1 << sh)) << (32 - sh))
        a.append(x); b.append(edit_ops(rng, y, int(rng.integers(0, 3))))
    a += rng.integers(0, 1 << 32, n_rand, dtype=np.uint64).tolist(); b += rng.integers(0, 1 << 32, n_rand, dtype=np.uint64).tolist()
    a = np.asarray(a, np.uint32); b = np.asarray(b, np.uint32)
    lo, hi = np.minimum(a, b), np.maximum(a, b)
    keep = lo != hi
    return lo[keep], hi[keep]


def oracle_D(a, b):
    L = orc.lib()
    return np.fromiter((min(L.orc_ed(int(x), 16, int(y), 16), L.orc_ed(int(x), 15, int(y), 16), L.orc_ed(int(x), 16, int(y), 15))
                        for x, y in zip(a, b)), np.int32, a.size)


def test_scheme_tables(shim):
    """Condition counts of the three layouts; keys fit the one-digit counting sort; the symmetric condition opens each set."""
    want = {5: (74, 10, 10), 6: (215, 20, 20), 7: (475, 35, 35)}
    for nb, (nc, ns, nsets) in want.items():
        assert use_layout(shim, nb) == nc
        assert (shim.shim3_nself(), shim.shim3_nsets()) == (ns, nsets)
        assert all(shim.shim3_key_bits(c) <= 20 for c in range(nc))
        firsts = [c for c in range(nc) if c == 0 or shim.shim3_set(c) != shim.shim3_set(c - 1)]
        assert len(firsts) == nsets and all(shim.shim3_self(c) for c in firsts)
        assert sum(shim.shim3_self(c) for c in range(nc)) == ns
    bad = (C.c_int * 7)(3, 2, 2, 2, 2, 3, 1)                       # a 1-base block: refused
    assert shim.shim3_scheme(bad, 7) == -1


@pytest.mark.parametrize("nb", [6, 7])
def test_necessity_and_handover_random_pairs(shim, nb):
    use_layout(shim, nb)
    a, b = near_pairs(11 + nb)
    D = oracle_D(a, b)
    slow = np.zeros(a.size, np.int32); fast = np.zeros(a.size, np.int32)
    shim.shim3_first(a, b, a.size, slow, fast)
    quick = np.zeros(a.size, np.uint8)
    shim.shim3_quick(a, b, a.size, quick)
    near = D <= 3
    assert near.sum() > 15000 and (D == 3).sum() > 3000
    assert (slow[near] != NONE).all(), "a pair with D <= 3 meets no condition"
    assert quick[near].all(), "the quick test rejects a pair with D <= 3"
    assert np.array_equal(fast, slow), "the kernel's hand-over differs from the definition"
    assert (slow[~near] != NONE).any() and (slow[~near] == NONE).any()


@pytest.mark.parametrize("nb", [6, 7])
def test_necessity_complete_neighbourhoods(shim, nb):
    """Every word within three edit operations of a few dozen random and repetitive 16-mers."""
    use_layout(shim, nb)
    rng = np.random.default_rng(3 + nb)
    seeds = [int(v) for v in rng.integers(0, 1 << 32, 16)] + [periodic(rng) for _ in range(16)] + [0, 0xFFFFFFFF, 0x55555555, 0x1B1B1B1B]
    out = (C.c_ulonglong * 5)()
    near = 0
    for w in seeds:
        shim.shim3_neighbourhood(w, 16, out)
        words, n3, missed, quick_fail, differ = list(out)
        assert missed == 0 and quick_fail == 0 and differ == 0, (hex(w), list(out))
        near += n3
    assert near > 1000000


def test_join_emulation_vs_oracle(shim):
    """The join passes with the kernel's own per-pair functions give exactly the oracle's edge set at t = 3."""
    use_layout(shim, 7)
    rng = synth.rng_for(5)
    sets = []
    cells = rng.integers(0, 1 << 32, 60, dtype=np.uint64).astype(np.uint32)
    obs, _ = synth.simulate_reads(cells, 4000, 0.08, rng)
    sets.append(np.unique(obs))
    base = int(rng.integers(0, 1 << 31))
    sets.append(np.unique(np.concatenate([np.arange(base, base + 600, dtype=np.uint64),
                                          (np.arange(0, 400, dtype=np.uint64) << np.uint64(20)) + np.uint64(0x55555)]).astype(np.uint32)))
    sets.append(np.unique(np.asarray([periodic(rng) for _ in range(300)] + [edit_ops(rng, periodic(rng), 2) for _ in range(300)], np.uint32)))
    for s in sets:
        cap = s.size * s.size
        oa = np.zeros(cap, np.uint32); ob = np.zeros(cap, np.uint32); od = np.zeros(cap, np.uint8)
        st = (C.c_ulonglong * 5)()
        n = shim.shim3_join_emulate(s, s.size, oa.ctypes.data, ob.ctypes.data, od.ctypes.data, cap, st)
        got = np.stack([oa[:n], ob[:n], od[:n]], 1).astype(np.int64)
        got = got[np.lexsort((got[:, 1], got[:, 0]))]
        wa, wb, wd, _ = orc.Index(s).edges(3)
        assert np.array_equal(got, np.stack([wa, wb, wd], 1).astype(np.int64))
        assert st[3] >= n and st[2] >= st[3] and n > 100
