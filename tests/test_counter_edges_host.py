"""tests/counter_geometry.py without a GPU: window_keys, the vectorised reference of the k-mer counter's table, equals
count_table at every k in both modes, and geometry / merge_geometry / host_chunks / scan_passes equal a brute-force
count of the same shapes on small batches."""
import bisect
import itertools
from collections import Counter

import numpy as np
import pytest

from oracle import oracle
from tests import counter_geometry as cg
from tests.test_counter_host import count_table, pack
from tests.test_gpu_hypothesis import ALPHABETS
from tests.util import random_batch


def alphabet_batch(rng, k):
    """Sequences from each of the dense tests' alphabets, with empty records between them and at both ends."""
    seqs = [b""]
    for name, alpha in sorted(ALPHABETS.items()):
        a = np.frombuffer(alpha, np.uint8)
        for n in (k - 1, k, 3 * k + 5, 300):
            seqs += [a[rng.integers(0, len(a), size=max(n, 0))].tobytes(), b""]
    return pack(seqs + [b"", b"N" * 40, b"ACGT" * 9, b""])


@pytest.mark.parametrize("k", range(1, 32))
def test_window_keys_equals_count_table(k):
    rng = np.random.default_rng(k)
    lens = [0, 0, 1, k - 1, k, k + 1, 2 * k, 0, 4095, 4097] + list(rng.integers(0, 500, size=30)) + [0]
    batches = [random_batch(rng, lens, noise=0.03, n_runs=0.4), alphabet_batch(rng, k)]
    b, o = batches[0]
    batches.append((np.concatenate([np.frombuffer(b"ACGTN" * 20, np.uint8), b]), o + 100))   # offsets[0] > 0
    for bases, offsets in batches:
        for canonical in (True, False):
            got = cg.window_keys(bases, offsets, k, canonical)
            want = count_table(bases[int(offsets[0]):], offsets - offsets[0], k, canonical)
            assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]) and got[2] == want[2]


def brute_windows(bases, offsets, k, canonical):
    """(end position relative to offsets[0], key) of every valid window, by the reference's rolling update."""
    nt4 = cg.nt4_table()
    mask = (1 << 2 * k) - 1
    out = []
    for i in range(len(offsets) - 1):
        f = r = run = 0
        for j in range(int(offsets[i]), int(offsets[i + 1])):
            c = int(nt4[bases[j]])
            if c < 4:
                f = ((f << 2) | c) & mask
                r = (r >> 2) | ((3 - c) << 2 * (k - 1))
                run += 1
            else:
                run = 0
            if run >= k:
                out.append((j - int(offsets[0]), min(f, r) if canonical else f))
    return out


@pytest.mark.parametrize("k,canonical", [(1, True), (4, False), (5, True), (12, False), (13, True), (31, False),
                                         (31, True)])
def test_geometry_equals_a_brute_force_count(k, canonical):
    rng = np.random.default_rng(50 + k)
    T = cg.CT_T
    lens = [0, 5, T - 3, 0, 0, 2 * T + 7, 1, k, 0, 3000, 9000] + [3] * 900 + [0]
    bases, offsets = random_batch(rng, lens, noise=0.01, n_runs=0.3)
    bases[int(offsets[5]) + 3000:int(offsets[6])] = ord("N")        # a whole tile without a valid window
    bases[:3000] = np.frombuffer(b"T", np.uint8)                    # keys 0xFF... in raw mode
    bases = np.concatenate([np.frombuffer(b"GATTACA" * 3, np.uint8), bases])
    offsets = offsets + 21
    W = int(offsets[-1] - offsets[0]) + 5000
    g = cg.geometry(bases, offsets, k, canonical, total_bases=W)
    win = brute_windows(bases, offsets, k, canonical)
    assert g.W == W and g.nt_k == -(-W // T)
    L = int(offsets[-1] - offsets[0])
    nt = -(-L // T)
    assert g.tiles.valid.tolist() == [sum(1 for p, _ in win if p // T == t) for t in range(nt)]
    rel = [int(x - offsets[0]) for x in offsets]
    assert g.tiles.inner.tolist() == [len({s for s in rel[:-1] if t * T < s < min((t + 1) * T, L)}) for t in range(nt)]
    assert 0 in g.tiles.valid and g.tiles.empty_at.tolist() == [rel[i] for i in range(len(rel) - 1) if rel[i] == rel[i + 1]]
    # the radix sort, pass by pass, as a stable Python sort
    keys = [key for _, key in win]
    nk, npass = len(keys), -(-2 * k // 8)
    r = g.radix
    assert (r.nk, r.nt_r, r.nv, r.passes, r.in_y) == (nk, -(-W // cg.RX_T), nk % cg.RX_T, npass, npass % 2 == 1)
    cur = list(keys)
    for p in range(npass):
        digits = [(x >> 8 * p) & 255 for x in cur]
        tiles = [digits[i:i + cg.RX_T] for i in range(0, nk, cg.RX_T)]
        assert r.digit_max[p] == max(max(Counter(t).values()) for t in tiles)
        assert r.tail_255[p] == (nk % cg.RX_T != 0 and 255 in tiles[-1])
        cur = sorted(cur, key=lambda x: (x >> 8 * p) & 255)
    assert cur == sorted(keys)
    if k <= 4 and not canonical:
        assert r.tail_255[0]
    passes, b0 = 0, 0
    while b0 < -(-cg.RX_DIGITS * r.nt_r // cg.SP_WB):
        passes, b0 = passes + 1, b0 + cg.SCAN_TOP
    assert r.scan_passes == passes
    # run-length encoding
    heads, at = [], 0
    for _, grp in itertools.groupby(cur):
        n = len(list(grp))
        heads.append((at, at + n))
        at += n
    ru = g.runs
    assert ru.nruns == len(heads) and ru.longest == max(e - h for h, e in heads)
    assert ru.block_cross == sum(h // cg.SP_WB != (e - 1) // cg.SP_WB for h, e in heads)
    assert ru.thread_cross == sum(h // 16 != (e - 1) // 16 for h, e in heads)
    assert ru.block_heads == sum(h % cg.SP_WB == 0 for h, _ in heads) and ru.last_len == heads[-1][1] - heads[-1][0]


def test_merge_geometry_equals_bisect():
    rng = np.random.default_rng(3)
    cases = [([], [1, 2]), ([1, 2], []), ([5, 9], [1, 2]), ([1, 2], [5, 9]), ([1, 3, 5], [2, 4, 6]), ([2, 4], [2, 4]),
             ([0, 7, 15], [7])]
    cases += [(np.unique(rng.integers(0, 60, size=rng.integers(0, 30))), np.unique(rng.integers(0, 60, size=rng.integers(0, 30))))
              for _ in range(40)]
    for a, b in cases:
        a, b = [int(x) for x in a], [int(x) for x in b]
        m = cg.merge_geometry(np.array(a, np.uint64), np.array(b, np.uint64))
        lb = [bisect.bisect_left(b, x) for x in a]
        ub = [bisect.bisect_right(a, x) for x in b]
        assert m == cg.Merge(len(a), len(b), len(set(a) & set(b)), 0 in lb, len(b) in lb, 0 in ub, len(a) in ub)


def test_host_chunks_is_the_cut_loop(monkeypatch):
    monkeypatch.setattr(cg, "HOST_CHUNK_BASES", 100)
    rng = np.random.default_rng(4)
    for _ in range(200):
        lens = rng.choice([0, 0, 1, 30, 99, 100, 101, 250], size=rng.integers(1, 20))
        off = np.r_[0, np.cumsum(lens)].astype(np.uint64)
        cut, i0, n = [], 0, len(lens)
        while i0 < n:   # the loop of ChunkPlan (host_common.h), as written there
            i1 = i0 + 1
            while i1 < n and off[i1 + 1] - off[i0] <= 100:
                i1 += 1
            cut.append((i0, i1, int(off[i1] - off[i0])))
            i0 = i1
        assert cg.host_chunks(off) == cut


def test_window_keys_at_scale_equals_the_oracle():
    """Block boundaries of window_keys (2^24 window ends) inside a sequence and across sequences."""
    rng = np.random.default_rng(6)
    bases, offsets = random_batch(rng, [(1 << 24) + 5, 3, 40_000], noise=0.001, n_runs=0.5)
    for k, canonical in ((1, True), (21, True), (31, False)):
        got = cg.window_keys(bases, offsets, k, canonical)
        f, r, _ = oracle.kmer_arrays(bases[:int(offsets[1])], k)
        rest = count_table(bases, offsets[1:] , k, canonical)
        u, c = np.unique(np.r_[np.minimum(f, r) if canonical else f, np.repeat(rest[0], rest[1].astype(np.int64))],
                         return_counts=True)
        assert np.array_equal(got[0], u) and np.array_equal(got[1], c.astype(np.uint64))
