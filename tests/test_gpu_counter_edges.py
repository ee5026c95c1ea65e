"""The batch-wide k-mer counter (ktb_counter_*, KmerCounter, `kmertools ctr`) at the edges of its index arithmetic: key
tiles, radix tiles and their padding, the histogram scan's carry loop, run blocks, merge shapes, host chunk cuts,
failed adds, reads in flight during an add and the output slices of `kmertools ctr`.

Every case asserts the shapes its batch was built for (tests/counter_geometry.py: geometry, merge_geometry,
host_chunks), so that a change to a generator cannot quietly stop reaching an edge, then compares keys, counts, len()
and .windows exactly with tests/test_counter_host.py::count_table or, for large batches, with
tests/counter_geometry.py::window_keys (checked against count_table on the CPU).

Heavy cases, on one B200: test_failed_host_add_leaves_the_table (about 6 Gbases of host input),
test_cli_output_slices (files of 8.4 M records), test_radix_scan_carry_loop and test_host_chunk_cuts (2^26 bases and
more per add)."""
from __future__ import annotations

import ctypes as C
import subprocess
from pathlib import Path

import numpy as np
import pytest
from hypothesis import HealthCheck, given, settings, strategies as st

from kmertools_b200 import KmerCounter, KtbError, _lib
from kmertools_b200.io import read_fastx
from tests import counter_geometry as cg
from tests.test_counter_host import count_table, pack
from tests.test_gpu_hypothesis import ALPHABETS
from tests.util import ALPHA, random_batch

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

ROOT = Path(__file__).resolve().parent.parent
BIN = ROOT / "kmertools_b200" / "bin" / "kmertools"
DEV = torch.device("cuda", 0)
T = cg.CT_T
CHUNK = cg.HOST_CHUNK_BASES


# ------------------------------------------------------------------------------------------------------------- helpers
def on_device(bases, offsets, dev=DEV):
    return (torch.from_numpy(np.require(bases, np.uint8, ["C", "W"])).to(dev),
            torch.from_numpy(np.asarray(offsets, dtype=np.int64)).to(dev))


def acgt(rng, n):
    return ALPHA[rng.integers(0, 4, size=n, dtype=np.uint8)]


def table(c):
    keys, counts = c.result()
    return keys, counts, c.windows, len(c)


def assert_table(c, want, what=""):
    keys, counts, windows, n = table(c)
    assert np.array_equal(keys, want[0]), f"{what}: keys differ"
    assert np.array_equal(counts, want[1]), f"{what}: counts differ"
    assert windows == want[2] and n == len(want[0]), f"{what}: windows {windows} / len {n}"


def add_device(c, tb, to, n, total, stream=None):
    """ktb_counter_add_device with an explicit total_bases: the return code."""
    s = stream if stream is not None else torch.cuda.current_stream(DEV)
    return _lib.load().ktb_counter_add_device(c._h, tb.data_ptr(), to.data_ptr(), n, total, s.cuda_stream)


def both_entries(bases, offsets, k, canonical, want, what=""):
    """A fresh counter per entry point: the host add, and add_tensors of the same batch."""
    with KmerCounter(k, canonical) as c:
        c.add((bases, offsets))
        assert_table(c, want, f"{what} host")
    with KmerCounter(k, canonical) as c:
        c.add_tensors(*on_device(bases, offsets))
        assert_table(c, want, f"{what} device")


def records(keys, k):
    """One record of exactly k bases per key: its ACGT text (first base most significant)."""
    keys = np.asarray(keys, dtype=np.uint64)
    shifts = np.uint64(2) * np.arange(k - 1, -1, -1, dtype=np.uint64)
    bases = ALPHA[((keys[:, None] >> shifts[None, :]) & np.uint64(3)).astype(np.int64)].reshape(-1)
    return bases, np.arange(len(keys) + 1, dtype=np.uint64) * np.uint64(k)


def rev_comp(keys, k):
    keys = np.asarray(keys, dtype=np.uint64)
    r = np.zeros_like(keys)
    for i in range(k):
        r = (r << np.uint64(2)) | (np.uint64(3) - ((keys >> np.uint64(2 * i)) & np.uint64(3)))
    return r


def merged(want, other):
    """The table of two reference tables added together."""
    keys = np.concatenate([want[0], other[0]])
    counts = np.concatenate([want[1], other[1]])
    u, inv = np.unique(keys, return_inverse=True)
    c = np.zeros(len(u), np.uint64)
    np.add.at(c, inv, counts)
    return u.astype(np.uint64), c, want[2] + other[2]


EMPTY = (np.zeros(0, np.uint64), np.zeros(0, np.uint64), 0)


# ----------------------------------------------------------------------------------------------------------- key tiles
TILE_STARTS = lambda k: sorted({x % T for x in (0, 1, k - 1, k, 30, 31, 32, T - k, T - k + 1, T - 1)})


def tile_batch(k, seed):
    """Sequences starting at every offset of TILE_STARTS(k) within a tile; an N run over the whole first tile, one over
    a middle tile and one over the last; a tile with all 4,096 windows valid; a tile of 4,096 one-base records; empty
    records on a tile's first and last byte."""
    rng = np.random.default_rng(seed)
    parts, pos = [], 0

    def put(seq):
        nonlocal pos
        parts.append(seq)
        pos += len(seq)

    put(b"N" * (T + 5))                                   # tile 0 has no valid window
    for o in TILE_STARTS(k):                              # a sequence starting at offset o of the next tile
        gap = (-pos) % T + o + T
        put(acgt(rng, gap).tobytes())
    put(b"")
    put(acgt(rng, (-pos) % T + 3 * T).tobytes())          # every window of its middle tiles valid
    put(b"")                                              # empty records on a tile's first byte
    put(b"")
    mid = acgt(rng, 2 * T + 300)
    mid[100:100 + 2 * T] = ord("N")                       # a middle tile without a valid window
    put(mid.tobytes())
    put(acgt(rng, (-pos) % T + T - 1).tobytes())
    put(b"")                                              # an empty record on a tile's last byte
    for _ in range(2 * T + 1):                            # a tile of one-base records
        put(bytes([int(ALPHA[rng.integers(0, 4)])]))
    put(acgt(rng, (-pos) % T + 100).tobytes())
    put(b"N" * (T + 1))                                   # the last tile has no valid window
    bases, offsets = pack(parts)
    return bases, offsets


def check_tile_geometry(g, offsets, k):
    rel = (np.asarray(offsets, np.int64) - int(offsets[0]))
    starts = set((rel[:-1][np.diff(rel) > 0] % T).tolist())
    assert set(TILE_STARTS(k)) <= starts
    v = g.tiles.valid
    assert v[0] == 0 and v[-1] == 0 and (v[1:-1] == 0).any() and (v == T).any()
    assert (g.tiles.inner == T - 1).any()                 # a tile of 4,096 one-base records
    e = g.tiles.empty_at % T
    assert (e == 0).any() and (e == T - 1).any()


@pytest.mark.parametrize("k", range(1, 32))
def test_key_tiles(k):
    bases, offsets = tile_batch(k, k)
    for canonical in (True, False):
        g = cg.geometry(bases, offsets, k, canonical, detail=False)
        check_tile_geometry(g, offsets, k)
        want = cg.window_keys(bases, offsets, k, canonical)
        both_entries(bases, offsets, k, canonical, want, f"k={k}")
        # device entry point: offsets[0] at residues 1, 4095 and 4096 + 30 of the buffer, total_bases = offsets[n] and
        # larger; the bytes around the batch are bases that must not be counted
        rng = np.random.default_rng(k + 100)
        for r in (1, T - 1, T + 30):
            buf = np.concatenate([acgt(rng, r), bases, acgt(rng, 777)])
            tb, to = on_device(buf, offsets + np.uint64(r))
            for total in (int(offsets[-1]) + r, len(buf)):
                with KmerCounter(k, canonical) as c:
                    _lib.check(add_device(c, tb, to, len(offsets) - 1, total))
                    assert_table(c, want, f"k={k} residue {r} total {total}")


# ---------------------------------------------------------------------------------------------------------- radix sort
@pytest.mark.parametrize("k", [5, 16, 31])
def test_radix_key_counts(k):
    """nk = 1, 4095, 4096, 4097 and m * 4096 - 1, m * 4096, m * 4096 + 1 valid windows in one sequence."""
    m = 7
    rng = np.random.default_rng(k)
    for nk in (1, T - 1, T, T + 1, m * T - 1, m * T, m * T + 1):
        bases, offsets = pack([acgt(rng, nk + k - 1).tobytes(), b"N" * 50])
        for canonical in (True, False):
            g = cg.geometry(bases, offsets, k, canonical)
            assert g.radix.nk == nk and g.radix.nv == nk % T
            both_entries(bases, offsets, k, canonical, count_table(bases, offsets, k, canonical), f"k={k} nk={nk}")


@pytest.mark.parametrize("k", [4, 8, 12, 16, 31])
def test_radix_tail_ties_the_padding(k):
    """Raw keys 0xFF... (T...T) fill the partial last tile: their digit is 255 in every pass whose digit has 8 key bits,
    the digit of the ~0 padding."""
    rng = np.random.default_rng(k)
    bases, offsets = pack([acgt(rng, 3 * T + k - 1 - 5).tobytes(), b"T" * (300 + k - 1), b"T" * (k + 40)])
    g = cg.geometry(bases, offsets, k, False)
    full = [p for p in range(g.radix.passes) if 8 * (p + 1) <= 2 * k]
    assert g.radix.nv == (3 * T - 5 + 300 + 41) % T and g.radix.nv > 300
    assert all(g.radix.tail_255[p] for p in full) and full
    both_entries(bases, offsets, k, False, count_table(bases, offsets, k, False), f"k={k}")


@pytest.mark.parametrize("k", [8, 16])
def test_radix_one_digit_then_all_digits(k):
    """Tiles whose 4,096 keys share one digit in every pass but the last, and spread over all 256 digits in the last."""
    rng = np.random.default_rng(k)
    top = 2 * k - 8
    keys = []
    for t in range(3):
        low = int(rng.integers(0, 1 << top))
        keys.append((np.arange(T, dtype=np.uint64) % np.uint64(256)) << np.uint64(top) | np.uint64(low))
    keys = np.concatenate(keys)
    bases, offsets = records(keys, k)
    g = cg.geometry(bases, offsets, k, False)
    assert g.radix.digit_max[:-1] == [T] * (g.radix.passes - 1) and g.radix.digit_max[-1] == T // 256
    want = count_table(bases, offsets, k, False)
    both_entries(bases, offsets, k, False, want, f"k={k}")


def test_radix_tiles_without_keys():
    """W far above nk: 10^6 reads of length k, and mostly-N input; most radix tiles hold no key."""
    rng = np.random.default_rng(1)
    k = 21
    bases, offsets = random_batch(rng, [k] * 1_000_000)
    g = cg.geometry(bases, offsets, k, True, detail=False)
    assert g.radix.nk == 1_000_000 and g.radix.nt_r > 20 * -(-g.radix.nk // T)
    both_entries(bases, offsets, k, True, cg.window_keys(bases, offsets, k), "reads of length k")
    bases = np.full(20_000_000, ord("N"), np.uint8)
    for i in range(0, len(bases), 1_000_003):
        bases[i:i + 60] = acgt(rng, 60)[:len(bases[i:i + 60])]
    offsets = np.array([0, 7_000_000, len(bases)], np.uint64)
    for canonical in (True, False):
        g = cg.geometry(bases, offsets, k, canonical, detail=False)
        assert 0 < g.radix.nk < 1000 and g.radix.nt_r > 4000
        both_entries(bases, offsets, k, canonical, cg.window_keys(bases, offsets, k, canonical), "mostly N")


def test_radix_scan_carry_loop():
    """One device add each of 2^26 and 2^26 + 1 bases: one and two passes of the digit matrix scan's carry loop."""
    rng = np.random.default_rng(2)
    k = 7
    base = acgt(rng, CHUNK + 1)
    base[::1000] = ord("N")
    for W in (CHUNK, CHUNK + 1):
        bases, offsets = base[:W], np.array([0, 12345, W], np.uint64)
        assert cg.scan_passes(cg.RX_DIGITS * -(-W // cg.RX_T)) == (1 if W == CHUNK else 2)
        want = cg.window_keys(bases, offsets, k)
        with KmerCounter(k) as c:
            c.add_tensors(*on_device(bases, offsets))
            assert_table(c, want, f"W={W}")


# ---------------------------------------------------------------------------------------------------------------- runs
RUN_LENGTHS = [T, T, 1, 15, 16, 17, 4095, 4096, 4097, 3 * T + 1, 1, 1, 16, 16, 15, 17]


@pytest.mark.parametrize("tail", [0, 1])
def test_runs(tail):
    """Runs of 1, 15, 16, 17, 4095, 4096, 4097 and 3 * 4096 + 1 equal keys, heads on a block's first entry, and a last
    run ending at nk with nk mod 4096 = tail; then one run over everything."""
    k = 12
    rng = np.random.default_rng(tail)
    lens = list(RUN_LENGTHS)
    lens.append(((tail - sum(lens)) % T) or T)
    keys = np.sort(rng.choice(4 ** k, size=len(lens), replace=False)).astype(np.uint64)
    rec = np.repeat(keys, lens)
    rng.shuffle(rec)
    bases, offsets = records(rec, k)
    g = cg.geometry(bases, offsets, k, False)
    assert g.radix.nk % T == tail and g.runs.nruns == len(lens) and g.runs.last_len == lens[-1]
    assert g.runs.block_heads >= 3 and g.runs.block_cross >= 4 and g.runs.thread_cross >= 8
    want = count_table(bases, offsets, k, False)
    assert sorted(want[1].tolist()) == sorted(lens)
    both_entries(bases, offsets, k, False, want, f"tail {tail}")
    for n in (2 * T + tail, 3 * T + 1):                   # a single run
        bases, offsets = records(np.full(n, keys[0]), k)
        g = cg.geometry(bases, offsets, k, False)
        assert g.runs.nruns == 1 and g.runs.longest == n
        both_entries(bases, offsets, k, False, count_table(bases, offsets, k, False), f"one run of {n}")


# -------------------------------------------------------------------------------------------------------------- merges
def test_merge_shapes():
    """A sequence of adds into one counter, each checked against the running reference and asserting its merge shape."""
    k = 6
    top = 4 ** k - 1
    rng = np.random.default_rng(3)
    even = np.arange(100, 2100, 2, dtype=np.uint64)
    steps = [
        ("empty table", even, lambda m: m.na == 0 and m.nb == len(even)),
        ("batch in table", even[::3], lambda m: m.dups == m.nb and m.na > m.nb),
        ("table in batch", np.r_[even, np.arange(2101, 2201, 2, dtype=np.uint64)], lambda m: m.dups == m.na < m.nb),
        ("equal sets", None, lambda m: m.dups == m.na == m.nb),
        ("interleaved", np.arange(101, 2100, 2, dtype=np.uint64), lambda m: m.dups == 0 and not m.ub0 and not m.ub_na),
        ("below", np.arange(10, 50, dtype=np.uint64), lambda m: m.dups == 0 and m.ub0 and not m.ub_na and m.lb_nb),
        ("above", np.arange(3000, 3100, dtype=np.uint64), lambda m: m.dups == 0 and m.ub_na and not m.ub0 and m.lb0),
        ("single below", np.array([0], np.uint64), lambda m: m.nb == 1 and m.ub0),
        ("single above", np.array([top], np.uint64), lambda m: m.nb == 1 and m.ub_na),
        ("ends", np.array([0, top], np.uint64), lambda m: m.nb == m.dups == 2),
    ]
    want = EMPTY
    with KmerCounter(k, False) as c:
        for i, (name, keys, shape) in enumerate(steps):
            if keys is None:
                keys = want[0]
            rec = np.repeat(keys, rng.integers(1, 4, size=len(keys)))
            rng.shuffle(rec)
            bases, offsets = records(rec, k)
            batch = count_table(bases, offsets, k, False)
            assert shape(cg.merge_geometry(want[0], batch[0])), name
            if i % 2:
                c.add_tensors(*on_device(bases, offsets))
            else:
                c.add((bases, offsets))
            want = merged(want, batch)
            assert_table(c, want, name)
        # bases but no valid window, into a non-empty table: nb = 0 with W > 0
        for bases, offsets in (pack(["N" * 5000, "ACGTA", "", "AC" + "N" * 9000]), pack(["ACG"] * 3000)):
            assert cg.geometry(bases, offsets, k, False).radix.nk == 0 and offsets[-1] > 0
            c.add((bases, offsets))
            assert_table(c, want, "no window, host")
            c.add_tensors(*on_device(bases, offsets))
            assert_table(c, want, "no window, device")


def test_merge_past_the_grid():
    """A table and a batch larger than the grids of count_merge_write_kernel and count_merge_dup_kernel (148 * 16 CTAs
    of 256 threads), so that both grid-stride loops turn."""
    rng = np.random.default_rng(4)
    k = 31
    n = cg.MERGE_GRID + 100_000
    first = random_batch(rng, [n // 2, n // 2 + 50])
    second = random_batch(rng, [n + 7])
    second[0][: n // 3] = first[0][: n // 3]   # a third of the batch is in the table
    want = cg.window_keys(*first, k)
    assert len(want[0]) > cg.MERGE_GRID
    with KmerCounter(k) as c:
        c.add_tensors(*on_device(*first))
        assert_table(c, want, "first")
        b = cg.window_keys(*second, k)
        m = cg.merge_geometry(want[0], b[0])
        assert m.nb > cg.MERGE_GRID and m.na + m.nb > cg.MERGE_GRID and m.dups > 100_000
        c.add((second[0], second[1]))
        assert_table(c, merged(want, b), "second")


@settings(max_examples=100, deadline=None, suppress_health_check=list(HealthCheck))
@given(data=st.data())
def test_random_add_sequences(data):
    k = data.draw(st.integers(1, 31))
    canonical = data.draw(st.booleans())
    seed = data.draw(st.integers(0, 2 ** 32 - 1))
    rng = np.random.default_rng(seed)
    want = EMPTY
    with KmerCounter(k, canonical) as c:
        for _ in range(data.draw(st.integers(1, 6))):
            alpha = np.frombuffer(ALPHABETS[data.draw(st.sampled_from(sorted(ALPHABETS)))], np.uint8)
            lens = data.draw(st.lists(st.sampled_from([0, 1, k - 1, k, k + 1, 2 * k, 100, T - 1, T, T + 1, 2 * T + 3]),
                                      min_size=1, max_size=12))
            lens = [max(x, 0) for x in lens]
            offsets = np.r_[0, np.cumsum(lens)].astype(np.uint64)
            bases = alpha[rng.integers(0, len(alpha), size=int(offsets[-1]))]
            if data.draw(st.booleans()):
                c.add((bases, offsets))
            else:
                c.add_tensors(*on_device(bases, offsets))
            want = merged(want, count_table(bases, offsets, k, canonical))
            assert_table(c, want)


# --------------------------------------------------------------------------------------------------------- host chunks
def chunk_batch(lens, rng):
    offsets = np.r_[0, np.cumsum(lens)].astype(np.uint64)
    bases = acgt(rng, int(offsets[-1]))
    bases[::997] = ord("N")
    return bases, offsets


@pytest.mark.parametrize("case", ["exact_chunk_then_one", "single_sequences", "empty_chunks"])
def test_host_chunk_cuts(case):
    """Chunk cuts of the host entry point against the device entry point and window_keys."""
    rng = np.random.default_rng(5)
    if case == "exact_chunk_then_one":
        lens, cuts = [CHUNK - 1000, 1000, 1], [(0, 2, CHUNK), (2, 3, 1)]
    elif case == "single_sequences":
        lens, cuts = [5, CHUNK, CHUNK + 1, 7], [(0, 1, 5), (1, 2, CHUNK), (2, 3, CHUNK + 1), (3, 4, 7)]
    else:   # chunks without bases before a sequence longer than a chunk and after it, beside a copy in flight
        lens, cuts = [0, 0, 0, CHUNK + 10, 0, 0], [(0, 3, 0), (3, 4, CHUNK + 10), (4, 6, 0)]
    bases, offsets = chunk_batch(lens, rng)
    assert cg.host_chunks(offsets) == cuts
    k, canonical = {"exact_chunk_then_one": (11, True), "single_sequences": (12, False), "empty_chunks": (11, False)}[case]
    want = cg.window_keys(bases, offsets, k, canonical)
    with KmerCounter(k, canonical) as h, KmerCounter(k, canonical) as d:
        h.add((bases, offsets))
        d.add_tensors(*on_device(bases, offsets))
        assert_table(h, want, f"{case} host")
        assert_table(d, want, f"{case} device")
    with KmerCounter(31) as h, KmerCounter(31) as d:
        h.add((bases, offsets))
        d.add_tensors(*on_device(bases, offsets))
        a, b = table(h), table(d)
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) and a[2:] == b[2:]


def test_host_offsets_not_at_zero_and_bad_offsets():
    """offsets[0] > 0 on the host entry point over several chunks; non-monotone offsets after earlier adds are
    KTB_ERR_ARG and leave the table as it was."""
    rng = np.random.default_rng(6)
    bases, offsets = chunk_batch([1000] + [40_000] * 1700 + [3], rng)
    sub = offsets[1:]
    assert sub[0] > 0 and len(cg.host_chunks(sub)) == 2
    k = 9
    want = cg.window_keys(bases, sub, k)
    with KmerCounter(k) as c:
        c.add((bases, sub))
        assert_table(c, want, "offsets[0] > 0")
        before = table(c)
        L = _lib.load()
        bad = sub.copy()
        bad[1000] = bad[999] - np.uint64(1)
        assert L.ktb_counter_add(c._h, bases.ctypes.data, bad.ctypes.data, len(bad) - 1) == _lib.KTB_ERR_ARG
        assert b"non-decreasing" in L.ktb_last_error()
        after = table(c)
        assert all(np.array_equal(x, y) for x, y in zip(before[:2], after[:2])) and before[2:] == after[2:]
        c.add((bases, sub))
        assert_table(c, merged(want, want), "after the error")


# ----------------------------------------------------------------------------------------------------- failed adds
def test_failed_device_add_leaves_the_table():
    """total_bases of 0x7fffffff key tiles: a scratch of 33 B a base that cannot be allocated (KTB_ERR_NOMEM); one tile
    more: "batch too large" (KTB_ERR_ARG).  The table, len() and .windows stay identical, and the next add works."""
    rng = np.random.default_rng(7)
    bases, offsets = random_batch(rng, [300, 40, 1000])
    tb, to = on_device(bases, offsets)
    want = count_table(bases, offsets, 15)
    L = _lib.load()
    with KmerCounter(15) as c:
        c.add_tensors(tb, to)
        before = table(c)
        for total, code in ((0x7FFFFFFF * T, _lib.KTB_ERR_NOMEM), (0x7FFFFFFF * T + 1, _lib.KTB_ERR_ARG)):
            assert add_device(c, tb, to, len(offsets) - 1, total) == code, L.ktb_last_error()
            after = table(c)
            assert all(np.array_equal(x, y) for x, y in zip(before[:2], after[:2])) and before[2:] == after[2:]
        torch.cuda.synchronize()
        c.add_tensors(tb, to)
        assert_table(c, merged(want, want), "after the errors")


def mem_available():
    with open("/proc/meminfo") as f:
        for line in f:
            if line.startswith("MemAvailable:"):
                return int(line.split()[1]) * 1024
    return 0


def test_failed_host_add_leaves_the_table():
    """A host add of a small chunk and then one sequence whose scratch exceeds the device's memory (about 6 Gbases on
    a B200): KTB_ERR_NOMEM, and the table the add started from is intact, not holding the first chunk."""
    total_mem = torch.cuda.get_device_properties(DEV).total_memory
    big = -(-int(1.05 * total_mem) // cg.SCRATCH_PER_BASE)
    if mem_available() < 2 * big:
        pytest.skip(f"needs {2 * big / 2**30:.0f} GiB of free host memory")
    rng = np.random.default_rng(8)
    small, so = random_batch(rng, [5000, 700])
    k = 21
    with KmerCounter(k) as c:
        c.add((small, so))
        before = table(c)
        bases = np.full(5700 + big, ord("A"), np.uint8)
        bases[:5700] = small
        offsets = np.array([0, 5000, 5700, 5700 + big], np.uint64)
        assert [x[2] for x in cg.host_chunks(offsets)] == [5700, big]
        with pytest.raises(KtbError) as e:
            c.add((bases, offsets))
        assert e.value.code == _lib.KTB_ERR_NOMEM
        del bases
        after = table(c)
        assert all(np.array_equal(x, y) for x, y in zip(before[:2], after[:2])) and before[2:] == after[2:]
        c.add((small, so))
        keys, counts, windows, _ = table(c)
        assert np.array_equal(keys, before[0]) and np.array_equal(counts, 2 * before[1]) and windows == 2 * before[2]


# --------------------------------------------------------------------------------------------------- reads then adds
def test_reads_are_ordered_before_the_next_add():
    """result_tensors() behind about a second of work on torch's current stream, then an add: the add returns only after the
    copies, which hold the table from before the add.  Host add of two chunks, then add_tensors on a second stream."""
    rng = np.random.default_rng(9)
    k = 13
    first = random_batch(rng, [10_000, 300])
    second = random_batch(rng, [CHUNK - 5, 3000])
    assert len(cg.host_chunks(second[1])) == 2
    s2 = torch.cuda.Stream(DEV)
    tb, to = on_device(*second)
    nwin = len(cg.position_keys(*second, k)[0])
    with KmerCounter(k) as c:
        c.add(first)
        for step in ("host", "device"):
            before = table(c)
            torch.cuda._sleep(2_000_000_000)
            keys, counts = c.result_tensors()
            ev = torch.cuda.Event()
            ev.record()
            if step == "host":
                c.add(second)
            else:
                with torch.cuda.stream(s2):
                    c.add_tensors(tb, to)
            assert ev.query(), f"{step}: the add returned before the copies of result_tensors ran"
            torch.cuda.synchronize()
            assert np.array_equal(keys.cpu().numpy().astype(np.uint64), before[0])
            assert np.array_equal(counts.cpu().numpy().astype(np.uint64), before[1])
            assert c.windows == before[2] + nwin


# ----------------------------------------------------------------------------------------------------- kmertools ctr
def ctr(*args, **kw):
    return subprocess.run([str(BIN), "ctr", *map(str, args)], capture_output=True, **kw)


def fasta(bases, offsets):
    n = len(offsets) - 1
    k = int(offsets[1] - offsets[0]) if n else 0
    rows = np.empty((n, k + 3), np.uint8)
    rows[:, 0], rows[:, 1], rows[:, -1] = ord(">"), ord("\n"), ord("\n")
    rows[:, 2:-1] = bases.reshape(n, k)
    return rows.tobytes()


def count_lines(keys, counts, k, acgt_text):
    if acgt_text:
        b, _ = records(keys, k)
        rows = np.empty((len(keys), k + 1), np.uint8)
        rows[:, :k] = b.reshape(len(keys), k)
        rows[:, k] = ord("\t")
        return b"".join(r + b"%d\n" % x for r, x in zip(map(bytes, rows), counts.tolist()))
    return "".join(f"{a}\t{b}\n" for a, b in zip(keys.tolist(), counts.tolist())).encode()


def test_cli_output_slices(tmp_path):
    """k = 31 with 2^22 - 1, 2^22, 2^22 + 1 and 2 * 2^22 + 1 distinct keys, one record of k bases per key and some
    records twice: the slice edges of the write-out, and more records than a parse batch holds."""
    k = 31
    rng = np.random.default_rng(10)
    pool = rng.integers(0, 4 ** k, size=int(2.2 * 2 * cg.SLICE), dtype=np.uint64)
    pool = np.unique(np.minimum(pool, rev_comp(pool, k)))
    rng.shuffle(pool)
    for n in (cg.SLICE - 1, cg.SLICE, cg.SLICE + 1, 2 * cg.SLICE + 1):
        keys = pool[:n]
        rec = np.r_[keys, keys[:5000]]
        bases, offsets = records(rec, k)
        src = tmp_path / "in.fa"
        src.write_bytes(fasta(bases, offsets))
        u = np.sort(keys)
        counts = np.ones(n, np.uint64)
        counts[np.searchsorted(u, keys[:5000])] = 2
        runs = [(3, False)] if n != cg.SLICE + 1 else [(1, False), (3, False), (64, False), (3, True), (64, True)]
        if n == 2 * cg.SLICE + 1:
            assert len(rec) > cg.MAX_RECORDS
        expected = {text: count_lines(u, counts, k, text) for text in {t for _, t in runs}}
        for threads, text in runs:
            out = tmp_path / "o"
            r = ctr("-i", src, "-o", out, "-k", k, "-t", threads, *(["--acgt"] if text else []))
            assert r.returncode == 0 and r.stderr == b"", r.stderr
            got = (out / "kmers.counts").read_bytes()
            assert got == expected[text], f"n={n} -t {threads} acgt={text}"
        if n == cg.SLICE + 1:   # ktb_count_file's stats
            st_ = _lib.FileStats()
            o = _lib.FileOpts(str(src).encode(), str(tmp_path / "s").encode(), k, 1, 0, b"\t", 0, 4, 0)
            _lib.check(_lib.load().ktb_count_file(C.byref(o), 0, C.byref(st_)))
            assert (st_.records, st_.bases) == (len(rec), len(rec) * k)
            assert st_.bytes_written == (tmp_path / "s" / "kmers.counts").stat().st_size > 0


@pytest.mark.parametrize("k", range(1, 10))
def test_cli_any_k(golden, tmp_path, k):
    bases, offsets = read_fastx(golden / "reads.fq")
    keys, counts, _ = count_table(bases, offsets, k)
    r = ctr("-i", golden / "reads.fq", "-o", tmp_path, "-k", k, "--any-k")
    assert r.returncode == 0 and r.stderr == b"", r.stderr
    assert (tmp_path / "kmers.counts").read_bytes() == count_lines(keys, counts, k, False)


def test_cli_empty_all_n_and_stdin(golden, tmp_path):
    for name, text in (("empty.fa", b""), ("alln.fa", b">a\nNNNNNNNNNNNNNNNNNNNNNNNNNNNNNNNNNNNNNNNNNNNN\n>b\n\n")):
        (tmp_path / name).write_bytes(text)
        r = ctr("-i", tmp_path / name, "-o", tmp_path / name[:-3], "-k", 11)
        assert r.returncode == 0 and r.stderr == b"", r.stderr
        assert (tmp_path / name[:-3] / "kmers.counts").read_bytes() == b""
    for fname in ("reads.fa", "reads.fq"):
        bases, offsets = read_fastx(golden / fname)
        keys, counts, _ = count_table(bases, offsets, 17)
        r = ctr("-i", "-", "-o", tmp_path / fname, "-k", 17, input=(golden / fname).read_bytes())
        assert r.returncode == 0 and r.stderr == b"", r.stderr
        assert (tmp_path / fname / "kmers.counts").read_bytes() == count_lines(keys, counts, 17, False)


def test_second_device(golden, tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("one GPU visible")
    dev1 = torch.device("cuda", 1)
    rng = np.random.default_rng(11)
    bases, offsets = random_batch(rng, list(rng.integers(0, 3000, size=300)) + [T + 1], noise=0.02)
    want = count_table(bases, offsets, 19)
    with KmerCounter(19, device=1) as c:
        c.add((bases, offsets))
        c.add_tensors(*on_device(bases, offsets, dev1))
        w2 = merged(want, want)
        assert_table(c, w2, "device 1")
        keys, counts = c.result_tensors()
        assert keys.device == dev1
        assert np.array_equal(keys.cpu().numpy().astype(np.uint64), w2[0])
        assert np.array_equal(counts.cpu().numpy().astype(np.uint64), w2[1])
    bases, offsets = read_fastx(golden / "reads.fa")
    keys, counts, _ = count_table(bases, offsets, 21)
    r = ctr("-i", golden / "reads.fa", "-o", tmp_path, "-k", 21, "--device", 1)
    assert r.returncode == 0 and r.stderr == b"", r.stderr
    assert (tmp_path / "kmers.counts").read_bytes() == count_lines(keys, counts, 21, False)
