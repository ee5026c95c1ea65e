"""Sparse (CSR) k-mer count rows at the edges of their index arithmetic (csrc/sparse_kernels.cuh, csrc/sparse.cu): every
piece width of the tile sort, merge shapes of 2 ... 129 tiles, the carry loop of the u64 scans, `cap` in the write-out of
both entry points, host chunks with a sequence of its own and an empty last chunk, and random batches at every k.

Every case asserts the tile and chunk shapes it was built for (tile_geometry, piece_keys, host_chunks), so that a change
to a generator cannot quietly stop reaching a branch, and compares row_ptr, codes, values (as bytes) and totals bit for
bit with tests/sparse_ref.py::sparse_rows, or, for batches of millions of reads, with padded_rows below, which is itself
checked against sparse_rows."""
from __future__ import annotations

import functools
from collections import namedtuple

import numpy as np
import pytest
from hypothesis import HealthCheck, given, settings, strategies as st

from kmertools_b200 import OligoComputer, _lib, kmer_counts
from oracle import oracle
from tests.counter_geometry import HOST_CHUNK_BASES, host_chunks
from tests.sparse_ref import scatter, sparse_rows
from tests.test_gpu_hypothesis import ALPHABETS
from tests.test_gpu_sparse import COMBOS, DT, _dev_rows, _finish
from tests.util import ALPHA, random_batch

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

T = 4096                     # SP_T (sparse_kernels.cuh): window-end positions per tile
SP_WB = 4096                 # SP_WB (sparse_kernels.cuh): entries per block of the scans and the count / write passes
SCAN_TOP = 1024              # block sums sparse_scan_top_kernel (sparse_kernels.cuh) scans per pass of its carry loop
SCAN_PASS = SCAN_TOP * SP_WB                      # 4,194,304 sequences: one pass of the carry loop
SENT = np.uint64(0xFFFF_FFFF_FFFF_FFF7)          # above every code (< 4^31), offset and total of these batches
VSENT = {0: np.uint32(0xFFFF_FFF9), 1: np.float32(-7.5), 2: np.float64(-7.25)}


# ------------------------------------------------------------------------------------------------------------ geometry
Span = namedtuple("Span", "a b m rounds half zero_start")
Geometry = namedtuple("Geometry", "np passes spans")


def sp_rounds(m: int) -> int:
    """Merge rounds of a sequence over m tiles: ceil(log2 m), as sp_rounds."""
    return (int(m) - 1).bit_length()


def sort_bits(k: int, np_: int) -> int:
    """Bits of the tile sort key (piece << 2k) | key: np_ is also the piece value of invalid windows."""
    return 2 * k + int(np_).bit_length()


def high_digits(k: int, np_: int) -> int:
    """4-bit digits of the tile sort read at bit b >= 64, where sp_digit takes the key's bits as 0."""
    return len(range(64, sort_bits(k, np_), 4)) if sort_bits(k, np_) > 64 else 0


def tile_geometry(offsets, k: int) -> Geometry:
    """The shapes sparse_tile_kernel and sparse_merge_kernel see for a batch (offsets[0] = the batch's first base).

    np[t]: pieces of tile t, 1 + the distinct sequence starts strictly inside it (empty records share a start byte).
    passes[t]: 4-bit LSD passes over sort_bits(k, np[t]); an odd count leaves the sorted keys in the second buffer.
    spans[s], for each sequence over m >= 2 tiles: its first and last tile a, b, m, its merge rounds, the pool half its
    final list lies in (rounds & 1), and whether its START piece has no window: it starts fewer than k positions before
    the end of tile a, so tail_start = nruns and the START group is empty."""
    off = np.asarray(offsets, dtype=np.int64) - int(offsets[0])
    total = int(off[-1])
    ts = np.arange(-(-total // T), dtype=np.int64) * T
    te = np.minimum(ts + T, total)
    starts = np.unique(off)
    npc = 1 + np.searchsorted(starts, te, "left") - np.searchsorted(starts, ts, "right")
    passes = np.array([-(-sort_bits(k, x) // 4) for x in npc], dtype=np.int64)
    nz = np.nonzero(np.diff(off))[0]
    a, b = off[nz] // T, (off[nz + 1] - 1) // T
    spans = {}
    for s, aa, bb in zip(nz[b > a], a[b > a], b[b > a]):
        m = int(bb - aa + 1)
        r = sp_rounds(m)
        spans[int(s)] = Span(int(aa), int(bb), m, r, r & 1, bool((aa + 1) * T - off[s] < k))
    return Geometry(npc, passes, spans)


def piece_keys(bases, offsets, k: int, canonical, s: int):
    """Distinct keys of sequence s's windows that end in each of its tiles: the run list of each of its pieces."""
    b0, start, stop = int(offsets[0]), int(offsets[s]), int(offsets[s + 1])
    out = []
    for x in range((start - b0) // T, (stop - 1 - b0) // T + 1):
        lo, hi = max(start, b0 + x * T - k + 1), min(stop, b0 + (x + 1) * T)
        f, r, _ = oracle.kmer_arrays(bases[lo:hi], k)
        out.append(np.unique(np.minimum(f, r) if canonical else f))
    return out


# ---------------------------------------------------------------------------------------------------------- references
@functools.lru_cache(maxsize=1)
def nt4_table():
    """The oracle's code of every byte value (4 = not a base)."""
    return np.array([oracle.nt4(b) for b in range(256)], dtype=np.uint8)


def padded_rows(bases, offsets, k: int, canonical=True, norm_mode: int = 0):
    """sparse_rows for batches of millions of short reads, vectorised: the reads padded to one width with code 4, f and r
    of every window from shifted code columns, the windows without a code 4 kept, and np.unique on row * 4^k + key."""
    off = np.asarray(offsets, dtype=np.int64)
    n, lens = len(off) - 1, np.diff(off)
    assert n * 4 ** k < 2 ** 63
    width = max(int(lens.max(initial=0)), k)
    codes = np.full((n, width), 4, dtype=np.uint8)
    row = np.repeat(np.arange(n), lens)
    codes[row, np.arange(len(row)) - np.repeat(off[:-1] - off[0], lens)] = nt4_table()[bases[off[0]:off[-1]]]
    nw = width - k + 1
    f = np.zeros((n, nw), np.uint64)
    r = np.zeros((n, nw), np.uint64)
    bad = np.zeros((n, nw), bool)
    for i in range(k):
        c = codes[:, i:i + nw]
        bad |= c == 4
        c = (c & 3).astype(np.uint64)
        f |= c << np.uint64(2 * (k - 1 - i))
        r |= (np.uint64(3) - c) << np.uint64(2 * i)
    ok = ~bad
    totals = ok.sum(axis=1).astype(np.uint64)
    key = (np.minimum(f, r) if canonical else f)[ok]
    u, cnt = np.unique(np.nonzero(ok)[0].astype(np.uint64) << np.uint64(2 * k) | key, return_counts=True)
    urow = (u >> np.uint64(2 * k)).astype(np.int64)
    row_ptr = np.zeros(n + 1, dtype=np.uint64)
    np.cumsum(np.bincount(urow, minlength=n), out=row_ptr[1:])
    values = cnt.astype(np.float64)
    if norm_mode:
        m = totals[urow].astype(np.float64)
        values /= np.maximum(1.0, 2 * m if (norm_mode == 2 and not canonical) else m)
    return row_ptr, u & np.uint64(4 ** k - 1), values, totals


def concat_rows(*parts):
    """The rows of consecutive sub-batches as the rows of one batch."""
    rp, base = [np.zeros(1, np.uint64)], np.uint64(0)
    for p in parts:
        rp.append(p[0][1:] + base)
        base += p[0][-1]
    return (np.concatenate(rp),) + tuple(np.concatenate([p[i] for p in parts]) for i in (1, 2, 3))


def slice_rows(want, n: int):
    """The rows of the first n sequences."""
    rp = want[0][:n + 1]
    return rp, want[1][:int(rp[-1])], want[2][:int(rp[-1])], want[3][:n]


def take_rows(got, rows):
    """The rows of the listed sequences, in that order."""
    rp, codes, vals, tot = got
    parts = [(np.array([0, rp[i + 1] - rp[i]], np.uint64), codes[int(rp[i]):int(rp[i + 1])],
              vals[int(rp[i]):int(rp[i + 1])], tot[i:i + 1]) for i in rows]
    return concat_rows(*parts)


def assert_rows(got, want, dtype, what=""):
    """row_ptr exactly, codes, values as bytes and totals bit for bit against reference rows (values in f64); a failure
    names the first row that differs."""
    rp, codes, vals, tot = got
    w_rp, w_codes, w_vals, w_tot = want
    wv = w_vals.astype(dtype)
    if vals.dtype == np.int32:    # u32 rows through a torch int32 buffer
        vals = vals.view(np.uint32)
    same = (len(rp) == len(w_rp) and np.array_equal(rp, w_rp) and np.array_equal(tot, w_tot)
            and np.array_equal(codes, w_codes) and vals.dtype == wv.dtype
            and np.array_equal(vals.view(np.uint8), wv.view(np.uint8)))
    if same:
        return
    bad = []
    if len(rp) == len(w_rp):
        bad += list(np.nonzero(rp[1:] != w_rp[1:])[0][:1]) + list(np.nonzero(tot != w_tot)[0][:1])
        m = min(len(codes), len(w_codes))
        d = np.nonzero((codes[:m] != w_codes[:m]) | (vals[:m].view(np.uint8).reshape(m, -1)
                                                      != wv[:m].view(np.uint8).reshape(m, -1)).any(axis=1))[0]
        if len(d):
            bad.append(int(np.searchsorted(w_rp, d[0], "right")) - 1)
    i = min(bad) if bad else None
    detail = "" if i is None else (f"; first bad row {i}: got {codes[int(rp[i]):int(rp[i + 1])][:8]} total {tot[i]}, "
                                   f"want {w_codes[int(w_rp[i]):int(w_rp[i + 1])][:8]} total {w_tot[i]}")
    raise AssertionError(f"{what}: rows differ{detail}")


# ------------------------------------------------------------------------------------------------------------- callers
def _tensors(bases, offsets, dev=0):
    d = torch.device("cuda", dev)
    return torch.from_numpy(bases).to(d), torch.from_numpy(np.asarray(offsets, dtype=np.int64)).to(d)


def device_rows(bases, offsets, k, canonical, norm, code, **kw):
    """One fenced call of the device entry point over a whole batch (tests/test_gpu_sparse.py::_dev_rows)."""
    tb, to = _tensors(bases, offsets)
    n = len(offsets) - 1
    return _finish(_dev_rows(tb, to, n, int(offsets[-1]), k, canonical, norm, code, **kw), n, kw.get("totals", True))


def host_rows(bases, offsets, k, canonical, norm, code, cap, totals=True, device=0, fence=64):
    """ktb_sparse_vectorise into numpy buffers fenced by sentinels.  Checks that row_ptr (and totals) are complete and
    that nothing outside them, and nothing of codes / values at or past cap, was written; returns rows trimmed to
    min(nnz, cap)."""
    offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
    n = len(offsets) - 1
    rp = np.full(n + 1 + 2 * fence, SENT, np.uint64)
    tt = np.full(n + 2 * fence, SENT, np.uint64)
    cd = np.full(cap + 2 * fence, SENT, np.uint64)
    vl = np.full(cap + 2 * fence, VSENT[code], DT[code])

    def at(a):
        return a.ctypes.data + fence * a.itemsize
    _lib.check(_lib.load().ktb_sparse_vectorise(
        bases.ctypes.data if bases.size else None, offsets.ctypes.data, n, k, canonical, norm, code, device, at(rp),
        at(cd) if cap else None, at(vl) if cap else None, cap, at(tt) if totals else None))
    assert np.all(rp[:fence] == SENT) and np.all(rp[fence + n + 1:] == SENT) and not np.any(rp[fence:-fence] == SENT)
    if totals:
        assert np.all(tt[:fence] == SENT) and np.all(tt[fence + n:] == SENT) and not np.any(tt[fence:fence + n] == SENT)
    else:
        assert np.all(tt == SENT)
    row_ptr = rp[fence:fence + n + 1]
    m = min(int(row_ptr[-1]), cap)
    assert np.all(cd[:fence] == SENT) and np.all(cd[fence + m:] == SENT)
    assert np.all(vl[:fence] == VSENT[code]) and np.all(vl[fence + m:] == VSENT[code])
    return row_ptr, cd[fence:fence + m], vl[fence:fence + m], tt[fence:fence + n]


def capped(want, cap):
    rp, codes, vals, tot = want
    return rp, codes[:cap], vals[:cap], tot


def pack(records):
    """bases / offsets of a list of uint8 arrays."""
    offsets = np.zeros(len(records) + 1, dtype=np.uint64)
    np.cumsum([len(r) for r in records], out=offsets[1:])
    bases = np.concatenate(records).astype(np.uint8) if offsets[-1] else np.zeros(0, np.uint8)
    return bases, offsets


# ------------------------------------------------------------------------------------------------ A. tile-sort widths
NP_TARGETS = [1, 2, 3, 4, 7, 8, 15, 16, 31, 32, 63, 64, 127, 128, 255, 256, 511, 512, 1023, 1024, 2047, 2048, 4095, 4096]


def piece_lengths(rng, np_: int, k: int):
    """np_ piece lengths that fill one tile: k ... k + 40 bases for the first, middle and last piece as far as the tile
    allows, the rest of the tile spread over every other piece, so that one-base pieces sit between pieces with
    windows."""
    lens = np.ones(np_, dtype=np.int64)
    spare = T - np_
    for i in sorted({0, np_ // 2, np_ - 1}):
        add = min(spare, int(rng.integers(k, k + 41)) - 1)
        lens[i] += add
        spare -= add
    grow = np.arange(1, np_ - 1, 2) if np_ > 3 else np.arange(np_)
    lens += np.bincount(rng.choice(grow, size=spare), minlength=np_)
    assert lens.sum() == T
    return lens


def np_batch(rng, k: int):
    """One tile per target piece count, back to back.  A tile's first piece continues the previous tile's last record
    or starts a record on the tile's first byte; empty records share start bytes with non-empty ones, on tile first
    bytes too, and close the batch."""
    lens = []
    for ti, np_ in enumerate(rng.permutation(NP_TARGETS)):
        pieces = list(piece_lengths(rng, int(np_), k))
        if ti and rng.random() < 0.5:
            lens[-1] += pieces.pop(0)          # the tile's piece 0 is the HEAD of a record from the previous tile
        elif rng.random() < 0.6:
            lens += [0] * int(rng.integers(1, 3))   # empty records on the tile's first byte
        for p in pieces:
            if rng.random() < 0.03:
                lens.append(0)
            lens.append(int(p))
    lens += [0, 0, 0]
    return random_batch(rng, lens, noise=0.01)


@pytest.mark.parametrize("canonical", [1, 0])
@pytest.mark.parametrize("k", range(1, 32))
def test_tile_sort_every_piece_width(k, canonical):
    rng = np.random.default_rng(100 * k + canonical)
    bases, offsets = np_batch(rng, k)
    geo = tile_geometry(offsets, k)
    assert int(offsets[-1]) == len(NP_TARGETS) * T
    assert sorted(geo.np.tolist()) == NP_TARGETS                 # piece widths 1 ... 13 bits, each at both ends
    assert set((geo.passes % 2).tolist()) == {0, 1}              # the sorted keys end in either buffer
    lens = np.diff(offsets.astype(np.int64))
    at_tile_start = (lens == 0) & (offsets[:-1] % T == 0) & (offsets[:-1] < offsets[-1])
    assert at_tile_start.any() and np.all(lens[-3:] == 0)         # empty records on a tile's first byte and at the end
    assert {int(x).bit_length() for x in geo.np} == set(range(1, 14))
    if k == 31:
        assert high_digits(k, 4096) == 3                          # sp_digit's b >= 64 branch with 13 piece bits
    assert any(s.m >= 2 for s in geo.spans.values())
    want = sparse_rows(bases, offsets, k, canonical, 0)
    assert_rows(kmer_counts((bases, offsets), k, bool(canonical), 0, np.uint32), want, np.uint32, f"k={k} u32")
    if k in (1, 12, 13, 31):
        for norm, code in [(1, 1), (2, 2)]:
            assert_rows(device_rows(bases, offsets, k, canonical, norm, code),
                        sparse_rows(bases, offsets, k, canonical, norm), DT[code], f"k={k} norm={norm}")


# ----------------------------------------------------------------------------------------------------- B. merge shapes
MS = [2, 3, 4, 5, 7, 8, 9, 15, 16, 17, 32, 33, 64, 65, 129]   # neighbours of different round-count parity
KINDS = ["p1", "p2", "p3", "p7", "pT1", "rand"]
UNITS = {"p1": b"G", "p2": b"CA", "p3": b"TAC", "p7": b"GATTACA"}


def start_offsets(k: int):
    """Starts in the first tile: 0, 1, T - k (one window in the tile), T - k + 1 and T - 1 (none: zero-run START)."""
    return sorted({o for o in (0, 1, T - k, T - k + 1, T - 1) if o < T})


def merge_batch(rng, k: int):
    """Sequences over m in MS tiles for every start offset, back to back: each starts in the tile where the one before
    it ends (or on the next tile's first byte when its offset is 0, so that the one before ends on the tile edge).  Then
    a contig of 8 tiles with N over its tiles 2, 3 and 4, a read and three empty records.  Content cycles through
    period-1, 2, 3 and 7 repeats, a repeat of period T + 1, and A/C noise with one G in the first tile and one T in the
    last.  Returns bases, offsets, the index of each planned sequence, its kind, and the index of the N contig."""
    plan = [(m, o) for o in start_offsets(k) for m in MS] + [(8, 5)]
    starts, tile = [], 0
    for i, (m, o) in enumerate(plan):
        starts.append(tile * T + o)
        nxt = plan[i + 1][1] if i + 1 < len(plan) else T // 2
        tile = tile + m - 1 if nxt > 0 else tile + m
    ends = starts[1:] + [tile * T + T // 2]
    records = [ALPHA[rng.integers(0, 4, starts[0])]] if starts[0] else []
    first = len(records)
    kinds = []
    for i, (s, e) in enumerate(zip(starts, ends)):
        kind = KINDS[i % len(KINDS)] if i < len(plan) - 1 else "nblock"
        if kind in UNITS:
            seq = np.resize(np.frombuffer(UNITS[kind], np.uint8), e - s)
        elif kind == "pT1":
            seq = np.resize(ALPHA[rng.integers(0, 4, T + 1)], e - s)
        elif kind == "rand":
            seq = np.frombuffer(b"AC", np.uint8)[rng.integers(0, 2, e - s)]
            head = (s // T + 1) * T - s          # positions in the first tile
            if head >= k:                        # G in a window that ends in the first tile
                seq[int(rng.integers(0, head - k + 1))] = ord("G")
            seq[int(rng.integers((e - 1) // T * T, e)) - s] = ord("T")   # T in the last tile
        else:
            seq = ALPHA[rng.integers(0, 4, e - s)]
            a = s // T
            seq[(a + 2) * T - 5 - s:(a + 5) * T + 5 - s] = ord("N")
        records.append(seq)
        kinds.append(kind)
    records += [ALPHA[rng.integers(0, 4, 150)]] + [np.zeros(0, np.uint8)] * 3
    bases, offsets = pack(records)
    return bases, offsets, list(range(first, first + len(plan))), kinds


@pytest.mark.parametrize("canonical", [1, 0])
@pytest.mark.parametrize("k", [1, 2, 11, 12, 13, 21, 31])
def test_merge_shapes(k, canonical):
    rng = np.random.default_rng(200 + 2 * k + canonical)
    bases, offsets, seqs, kinds = merge_batch(rng, k)
    geo = tile_geometry(offsets, k)
    spans = [geo.spans[s] for s in seqs]
    for m in MS:                                  # every m, with and without a window in the START piece
        assert {sp.zero_start for sp in spans if sp.m == m} == ({True, False} if k >= 2 else {False}), m
    mixed = [i for i in range(len(seqs) - 1) if spans[i].b == spans[i + 1].a and spans[i].half != spans[i + 1].half]
    assert len(mixed) >= 10                       # HEAD of one and START of the next in one tile, final lists apart
    edge = [i for i in range(1, len(seqs)) if int(offsets[seqs[i]]) % T == 0]
    assert edge and all(spans[i - 1].b + 1 == spans[i].a for i in edge)   # ends on a tile edge, the next starts on it
    want = sparse_rows(bases, offsets, k, canonical, 0)
    for i, (s, kind) in enumerate(zip(seqs, kinds)):
        if kind == "nblock":
            keys = piece_keys(bases, offsets, k, canonical, s)
            assert [len(x) for x in keys[2:5]] == [0, 0, 0] and all(len(x) for x in keys[:2] + keys[5:])
            assert np.all(bases[int(offsets[s]) + 2 * T:int(offsets[s]) + 5 * T] == ord("N"))
        elif kind == "rand" and k >= 3:           # a key only in the first tile, one only in the last
            keys = piece_keys(bases, offsets, k, canonical, s)
            if not spans[i].zero_start:
                assert len(np.setdiff1d(keys[0], np.concatenate(keys[1:])))
            assert len(np.setdiff1d(keys[-1], np.concatenate(keys[:-1])))
        elif kind != "rand":                      # repeats: neighbouring pieces share keys, so every merge makes holes
            keys = piece_keys(bases, offsets, k, canonical, s)
            if kind == "pT1":                     # whole tiles miss one key of the period each; a short edge piece
                keys = keys[1:-1]                 # may hold just the key its neighbour misses
            keys = [x for x in keys if len(x)]
            assert all(len(np.intersect1d(x, y)) for x, y in zip(keys, keys[1:]))
            if len(keys) > 1:
                assert sum(len(x) for x in keys) > int(want[0][s + 1] - want[0][s])
    assert_rows(kmer_counts((bases, offsets), k, bool(canonical), 0, np.uint32), want, np.uint32, f"k={k} host")
    norm, code = (1, 1) if canonical else (2, 2)
    want_n = sparse_rows(bases, offsets, k, canonical, norm)
    got = device_rows(bases, offsets, k, canonical, norm, code)
    assert_rows(got, want_n, DT[code], f"k={k} device")
    if k <= 12:                                   # scattered into dense rows: equal to ktb_oligo_vectorise's
        n = len(offsets) - 1
        rows = range(n) if k <= 2 else sorted({seqs[-1], seqs[MS.index(129)], seqs[0], seqs[1], seqs[len(MS) + 3]})
        sub_b, sub_o = pack([bases[int(offsets[i]):int(offsets[i + 1])] for i in rows])
        oc = OligoComputer(k)
        dense = oc.vectorise_packed(sub_b, sub_o, norm_mode=norm, mins=bool(canonical), dtype=DT[code])
        pos_map = oc.kmer_pos_maps()[0] if canonical else None
        oc.close()
        rp, cd, vl, _ = take_rows(got, rows)
        mine = scatter(rp, cd, vl, dense.shape[1], pos_map, dtype=DT[code])
        assert np.array_equal(mine.view(np.uint8), dense.view(np.uint8))


# ------------------------------------------------------------------------------------------------------ C. scan passes
NS = [SCAN_PASS, SCAN_PASS + 1, 3 * SCAN_PASS + 17]


def scan_passes(n: int) -> int:
    """Passes of sparse_scan_top_kernel's carry loop in an exclusive scan of n entries."""
    return -(-(-(-n // SP_WB)) // SCAN_TOP)


@pytest.fixture(scope="module")
def short_reads():
    """NS[-1] reads of 1 ... 12 bases from ACGTN, about 5 % of the records empty; the smaller batches are prefixes."""
    rng = np.random.default_rng(300)
    n = NS[-1]
    lens = rng.integers(1, 13, size=n)
    lens[rng.random(n) < 0.05] = 0
    offsets = np.zeros(n + 1, dtype=np.uint64)
    np.cumsum(lens, out=offsets[1:])
    bases = np.frombuffer(b"ACGTN", np.uint8)[rng.integers(0, 5, int(offsets[-1]), dtype=np.uint8)]
    return bases, offsets


@pytest.mark.parametrize("canonical", [1, 0])
def test_scan_carry_loop(short_reads, canonical):
    """row_ptr and the list offsets of n = 2^22, 2^22 + 1 and 3 * 2^22 + 17 sequences in one device call (one, two and
    four passes of the carry loop), and the same batch through the host entry point, whose first chunk holds more than
    2^22 sequences."""
    bases, offsets = short_reads
    k = 5
    sub_o = offsets[:20_001]
    sub_b = bases[:int(sub_o[-1])]
    for norm in (0, 2):                           # the vectorised reference restates sparse_rows
        assert_rows(padded_rows(sub_b, sub_o, k, canonical, norm), sparse_rows(sub_b, sub_o, k, canonical, norm),
                    np.float64, f"padded_rows norm={norm}")
    want = padded_rows(bases, offsets, k, canonical, 0)
    assert [scan_passes(n) for n in NS] == [1, 2, 4]
    tb, to = _tensors(bases, offsets)
    for n in NS:
        w = slice_rows(want, n)
        got = _finish(_dev_rows(tb, to, n, int(offsets[n]), k, canonical, 0, 0, cap=int(w[0][-1])), n)
        for j in range(1, n // SCAN_PASS + 1):
            at = slice(j * SCAN_PASS - 2, min(n, j * SCAN_PASS + 2) + 1)
            assert np.array_equal(got[0][at], w[0][at]), (n, j)
        assert_rows(got, w, np.uint32, f"device n={n}")
    del tb, to
    torch.cuda.empty_cache()
    cuts = [c[:2] for c in host_chunks(offsets)]
    assert len(cuts) >= 2 and max(i1 - i0 for i0, i1 in cuts) > SCAN_PASS
    assert_rows(kmer_counts((bases, offsets), k, bool(canonical), 0, np.uint32), want, np.uint32, "host")


# ------------------------------------------------------------------------------------------ D. write-out, device entry
@pytest.mark.parametrize("k,canonical,norm,code", [(21, 1, 0, 0), (17, 0, 1, 1), (31, 0, 2, 2)])
def test_write_out_cap_device_entry(k, canonical, norm, code):
    """A low-complexity 1 Mbp contig, whose merged list is mostly holes, among reads and empty records: every cap from
    1 to nnz + 1 around rows and write-out blocks, with d_totals NULL and total_bases above offsets[n] in some calls."""
    rng = np.random.default_rng(400 + k)
    lens = [150] + list(rng.integers(0, 300, size=200)) + [1_000_017] + list(rng.integers(0, 300, size=200)) + [0, 0]
    lens = np.array(lens)
    lens[rng.choice(np.r_[1:201, 202:len(lens)], size=30, replace=False)] = 0
    bases, offsets = random_batch(rng, lens, noise=0.01, n_runs=0.1)
    c = int(np.argmax(lens))
    lo, hi = int(offsets[c]), int(offsets[c + 1])
    bases[lo:hi] = np.resize(np.frombuffer(b"TAC", np.uint8), hi - lo)
    bases[lo + rng.choice(hi - lo, size=10, replace=False)] = ord("G")
    n = len(lens)
    assert (lens == 0).sum() >= 20
    want = sparse_rows(bases, offsets, k, canonical, norm)
    rp = want[0]
    nnz, mid = int(rp[-1]), n // 2
    row_c = int(rp[c + 1] - rp[c])
    assert sum(len(x) for x in piece_keys(bases, offsets, k, canonical, c)) > 2 * row_c   # mostly holes
    caps = [1, int(rp[1]), int(rp[mid]) - 1, int(rp[mid]) + 1, 4095, 4096, 4097, nnz - 1, nnz, nnz + 1]
    assert len(set(caps)) == len(caps) and min(caps) == 1 < int(rp[1]) and max(caps) == nnz + 1
    tb, to = _tensors(bases, offsets)
    for j, cap in enumerate(caps):
        totals, total = j % 3 != 1, int(offsets[-1]) + (4097 if j % 2 else 0)
        got = _finish(_dev_rows(tb, to, n, total, k, canonical, norm, code, cap=cap, totals=totals), n, totals)
        if not totals:
            got = got[:3] + (want[3],)
        assert_rows(got, capped(want, cap), DT[code], f"cap={cap} totals={totals} total_bases={total}")


def test_device_and_host_entry_without_bases():
    """n > 0 sequences, all empty (total_bases = 0): row_ptr and totals are zero and nothing else is written."""
    n = 1000
    offsets = np.zeros(n + 1, dtype=np.uint64)
    tb, to = _tensors(np.zeros(16, np.uint8), offsets)
    zero = (np.zeros(n + 1, np.uint64), np.zeros(0, np.uint64), np.zeros(0, np.float32), np.zeros(n, np.uint64))
    for totals in (True, False):
        got = _finish(_dev_rows(tb, to, n, 0, 21, 1, 1, 1, cap=64, totals=totals), n, totals)
        assert_rows(got if totals else got[:3] + (zero[3],), zero, np.float32, f"device totals={totals}")
    assert_rows(host_rows(np.zeros(0, np.uint8), offsets, 21, 1, 1, 1, 64), zero, np.float32, "host")
    got = host_rows(np.zeros(0, np.uint8), np.zeros(1, np.uint64), 21, 1, 1, 1, 0)   # n = 0
    assert np.array_equal(got[0], np.zeros(1, np.uint64)) and len(got[3]) == 0


# ---------------------------------------------------------------------------------- E. host entry: chunks and cap
@pytest.fixture(scope="module")
def chunked_batch():
    """Reads | one (2^26 + 5000)-base sequence | reads and empty records | the same sequence | three empty records: five
    host chunks, the second and fourth one sequence each, the last without bases.  The long sequence is a period-7
    repeat with 20,000 point changes.  Returns bases, offsets and the reference rows at k = 21, canonical, NORM_CLI."""
    rng = np.random.default_rng(500)
    k = 21
    big = np.resize(np.frombuffer(b"GATTACA", np.uint8), HOST_CHUNK_BASES + 5000)
    big[rng.choice(len(big), size=20_000, replace=False)] = ALPHA[rng.integers(0, 4, 20_000)]
    parts = []
    for lens in ([150] + list(rng.integers(0, 400, size=3000)), [0, 0] + list(rng.integers(0, 400, size=3000)) + [0]):
        b, o = random_batch(rng, lens, noise=0.01, n_runs=0.1)
        parts.append([b[int(o[i]):int(o[i + 1])] for i in range(len(lens))])
    records = parts[0] + [big] + parts[1] + [big] + [np.zeros(0, np.uint8)] * 3
    bases, offsets = pack(records)
    ref_big = sparse_rows(big, np.array([0, len(big)], np.uint64), k, True, 1)
    want = concat_rows(sparse_rows(*pack(parts[0]), k, True, 1), ref_big, sparse_rows(*pack(parts[1]), k, True, 1),
                       ref_big, sparse_rows(*pack([np.zeros(0, np.uint8)] * 3), k, True, 1))
    return bases, offsets, want


def test_host_entry_chunks_and_cap(chunked_batch):
    bases, offsets, want = chunked_batch
    k, cn, norm, code = 21, 1, 1, 1
    cuts = [c[:2] for c in host_chunks(offsets)]
    nb = [int(offsets[i1] - offsets[i0]) for i0, i1 in cuts]
    assert len(cuts) == 5 and cuts[1][1] - cuts[1][0] == 1 and cuts[3][1] - cuts[3][0] == 1
    assert nb[1] == nb[3] == HOST_CHUNK_BASES + 5000
    assert nb[4] == 0 and cuts[4][1] - cuts[4][0] == 3   # the empty last chunk
    rp = want[0]
    first = [int(rp[i0]) for i0, _ in cuts] + [int(rp[-1])]       # first entry of each chunk
    nnz = first[-1]
    assert first[4] == nnz and all(first[i + 1] - first[i] > 1000 for i in range(4))
    caps = [nnz + 5, nnz, first[1] + (first[2] - first[1]) // 2, first[2], first[3] + (first[4] - first[3]) // 3,
            first[1] - 1]
    for j, cap in enumerate(caps):
        totals = j != 2
        got = host_rows(bases, offsets, k, cn, norm, code, cap, totals=totals)
        if not totals:
            got = got[:3] + (want[3],)
        assert_rows(got, capped(want, cap), DT[code], f"cap={cap} totals={totals}")
    assert_rows(host_rows(bases, offsets, k, cn, norm, code, 0), capped(want, 0), DT[code], "cap=0")


@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs two visible GPUs")
def test_second_device_both_entry_points():
    """device=1 on the host entry point and the device entry point under torch.cuda.device(1); the caller's current
    device stays what it was."""
    rng = np.random.default_rng(600)
    bases, offsets = random_batch(rng, [0, 150, T + 3, 2 * T + 1, 7, 0], noise=0.01)
    want = sparse_rows(bases, offsets, 21, True, 1)
    torch.cuda.set_device(0)
    assert_rows(host_rows(bases, offsets, 21, 1, 1, 1, len(bases), device=1), want, np.float32, "host device=1")
    assert torch.cuda.current_device() == 0
    tb, to = _tensors(bases, offsets, dev=1)
    with torch.cuda.device(1):
        got = _finish(_dev_rows(tb, to, len(offsets) - 1, len(bases), 21, 1, 1, 1), len(offsets) - 1)
        assert torch.cuda.current_device() == 1
    assert torch.cuda.current_device() == 0
    assert_rows(got, want, np.float32, "device 1")


# ------------------------------------------------------------------------------------ F. random batches at every k
@st.composite
def sparse_batches(draw):
    k = draw(st.integers(1, 31))
    alpha = np.frombuffer(ALPHABETS[draw(st.sampled_from(sorted(ALPHABETS)))], dtype=np.uint8)
    nseq = draw(st.integers(1, 10))
    edge = sorted({max(0, e + d) for e in (0, k - 1, k, T - 1, T, T + 1, 2 * T + 1) for d in (-1, 0, 1)})
    lengths = draw(st.lists(st.one_of(st.sampled_from(edge), st.integers(0, 600), st.integers(0, 3 * T)),
                            min_size=nseq, max_size=nseq))
    rng = np.random.default_rng(draw(st.integers(0, 2 ** 32 - 1)))
    seqs = [alpha[rng.integers(0, len(alpha), size=n)] for n in lengths]
    if draw(st.booleans()):   # a homopolymer member
        i = draw(st.integers(0, nseq - 1))
        seqs[i] = np.full(len(seqs[i]), ord(draw(st.sampled_from("ACGTN"))), dtype=np.uint8)
    canonical = draw(st.integers(0, 1))
    norm, code = draw(st.sampled_from(COMBOS))
    entry = draw(st.sampled_from(["host", "device"]))
    return k, seqs, canonical, norm, code, entry


@settings(max_examples=200, deadline=None, suppress_health_check=list(HealthCheck), derandomize=True)
@given(sparse_batches())
def test_random_batches_match_sparse_rows(example):
    k, seqs, canonical, norm, code, entry = example
    bases, offsets = pack(seqs)
    want = sparse_rows(bases, offsets, k, canonical, norm)
    if entry == "host":
        got = host_rows(bases, offsets, k, canonical, norm, code, max(1, len(bases)), fence=8)
    else:
        got = device_rows(bases, offsets, k, canonical, norm, code, fence=8)
    assert_rows(got, want, DT[code], f"k={k} canonical={canonical} norm={norm} code={code} {entry}")
