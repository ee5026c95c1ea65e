"""The shapes the batch-wide k-mer counter (csrc/count_kernels.cuh, csrc/counter.cu, ktb_count_file in csrc/file_api.cu)
sees for a batch, restated in Python, and window_keys, an exact reference of its table vectorised with numpy for batches
of millions of bases.

A test builds a batch for one edge of the counter's index arithmetic, asserts with geometry() / merge_geometry() /
host_chunks() that the batch reaches it, then compares the GPU table with the reference.  The geometry is itself
checked against a brute-force count in tests/test_counter_edges_host.py."""
from __future__ import annotations

import functools
from collections import namedtuple

import numpy as np

from oracle import oracle

CT_T = 4096                  # CT_T (count_kernels.cuh): window ends per key tile
RX_T = 4096                  # RX_T: keys per radix tile
RX_DIGITS = 256              # 8-bit digits per radix pass
SP_WB = 4096                 # SP_WB (sparse_common.cuh): entries per block of the run-length kernels and of scan_u64
SP_WITEMS = 16               # SP_WITEMS: consecutive entries per thread of those kernels
SCAN_TOP = 1024              # block sums sparse_scan_top_kernel scans per pass of its carry loop
SCAN_PASS = SCAN_TOP * SP_WB                     # 2^22 entries: one pass of that loop
HOST_CHUNK_BASES = 1 << 26   # HOST_CHUNK_BASES (host_common.h): bases per chunk of the host entry points
SLICE = 1 << 22              # keys per output slice of ktb_count_file
MAX_RECORDS = 4 << 20        # records per parse batch of ktb_count_file
MERGE_GRID = 148 * 16 * 256  # threads of the grid-stride merge kernels on a 148-SM B200 (sms * 16 CTAs of 256)
SCRATCH_PER_BASE = 33        # bytes of scratch per base of one add (include/kmertools_b200.h)


@functools.lru_cache(maxsize=1)
def nt4_table():
    """The oracle's code of every byte value (4 = not a base)."""
    return np.array([oracle.nt4(b) for b in range(256)], dtype=np.uint8)


def _codes(bases, offsets):
    off = np.asarray(offsets, dtype=np.int64)
    return nt4_table()[np.asarray(bases, dtype=np.uint8)[int(off[0]):int(off[-1])]], off - off[0]


def _window_codes(c, k: int, canonical):
    """Forward and reverse-complement codes (r is None in raw mode) of the windows starting at 0 .. len(c) - k of a
    code array, built from windows of 1, 2, 4, 8 and 16 codes joined along the bits of k."""
    L = len(c)
    f = r = None
    n_f = 0                                  # codes in f
    pf, pr, m = c, (np.uint64(3) - c) if canonical else None, 1
    kk = k
    while kk:
        if kk & 1:
            if f is None:
                f, r, n_f = pf, pr, m
            else:
                n = L - n_f - m + 1
                f = (f[:n] << np.uint64(2 * m)) | pf[n_f:n_f + n]
                if canonical:
                    r = (pr[n_f:n_f + n] << np.uint64(2 * n_f)) | r[:n]
                n_f += m
        kk >>= 1
        if kk:
            n = L - 2 * m + 1
            pf = (pf[:n] << np.uint64(2 * m)) | pf[m:m + n]
            if canonical:
                pr = (pr[m:m + n] << np.uint64(2 * m)) | pr[:n]
            m *= 2
    return f[:L - k + 1], (r[:L - k + 1] if canonical else None)


def position_keys(bases, offsets, k: int, canonical=True, block: int = 1 << 24):
    """(pos, keys): every valid window's end position (relative to offsets[0]), ascending, and its key.  That is the
    order in which count_keys_kernel writes the keys.  A window is valid when its k codes are bases of one sequence:
    the run of bases ending at it, reset at every sequence start and every non-base, is at least k long."""
    codes, off = _codes(bases, offsets)
    L = len(codes)
    # r0[i]: first position of the run of bases that ends at i (i + 1 where i is not a base)
    v = np.where(codes == 4, np.arange(1, L + 1, dtype=np.int64), 0)
    starts = off[:-1][off[:-1] < L]
    np.maximum.at(v, starts, starts)
    r0 = np.maximum.accumulate(v) if L else v
    pos, keys = [], []
    for a in range(k - 1, L, block):
        b = min(L, a + block)
        f, r = _window_codes((codes[a - k + 1:b] & 3).astype(np.uint64), k, canonical)
        ok = r0[a:b] <= np.arange(a, b, dtype=np.int64) - (k - 1)
        pos.append(np.nonzero(ok)[0] + a)
        keys.append((np.minimum(f, r) if canonical else f)[ok])
    if not pos:
        return np.zeros(0, np.int64), np.zeros(0, np.uint64)
    return np.concatenate(pos), np.concatenate(keys)


def window_keys(bases, offsets, k: int, canonical=True):
    """(keys u64, counts u64, windows) as tests/test_counter_host.py::count_table returns them."""
    _, keys = position_keys(bases, offsets, k, canonical)
    if k <= 12:   # a dense histogram of 4^k bins is faster than sorting
        c = np.bincount(keys.astype(np.int64), minlength=4 ** k)
        u = np.flatnonzero(c)
        return u.astype(np.uint64), c[u].astype(np.uint64), int(keys.size)
    u, c = np.unique(keys, return_counts=True)
    return u.astype(np.uint64), c.astype(np.uint64), int(keys.size)


# ------------------------------------------------------------------------------------------------------------ geometry
Tiles = namedtuple("Tiles", "valid inner empty_at")
Radix = namedtuple("Radix", "nk nt_r nv passes in_y digit_max tail_255 scan_passes")
Runs = namedtuple("Runs", "nruns block_cross thread_cross longest block_heads last_len")
Geometry = namedtuple("Geometry", "W nt_k tiles radix runs")
Merge = namedtuple("Merge", "na nb dups lb0 lb_nb ub0 ub_na")


def scan_passes(n: int) -> int:
    """Passes of sparse_scan_top_kernel's carry loop in scan_u64 over n entries: ceil(ceil(n / SP_WB) / SCAN_TOP)."""
    return -(-n // SCAN_PASS)


def radix_order(keys, p: int):
    """The keys as pass p of the radix sort reads them: stably sorted by their low 8p bits."""
    if p == 0:
        return keys
    low = keys & np.uint64((1 << (8 * p)) - 1)
    return keys[np.argsort(low, kind="stable")]


def geometry(bases, offsets, k: int, canonical=True, total_bases: int | None = None, detail: bool = True) -> Geometry:
    """The shapes of one add of a batch (offsets[0] = the batch's first base on the tile grid).

    W: bases the scratch is sized from (total_bases of a device add, default offsets[n] - offsets[0]); nt_k key tiles.
    tiles.valid[t]: valid windows ending in tile t of the batch; tiles.inner[t]: distinct sequence starts strictly
    inside tile t; tiles.empty_at: relative start bytes of the empty records (several may share one).
    radix: nk keys, nt_r = ceil(W / RX_T) radix tiles, nv = nk mod RX_T keys in the partial last tile, ceil(2k / 8)
    passes; in_y: an odd pass count leaves the sorted keys in the second buffer.  With detail, digit_max[p] is the
    largest count of one digit in one tile in pass p and tail_255[p] whether the partial last tile holds a real key whose
    digit is 255, which ties with the ~0 padding.  scan_passes: carry-loop passes of the scan of the [256][nt_r] matrix.
    runs (with detail): run count, runs that cross a 4,096-entry block edge and a 16-entry thread edge, the longest run,
    run heads on a block's first entry and the length of the last run, which ends at nk."""
    off = np.asarray(offsets, dtype=np.int64)
    L = int(off[-1] - off[0])
    W = L if total_bases is None else int(total_bases)
    pos, keys = position_keys(bases, offsets, k, canonical)
    nt = -(-L // CT_T)
    valid = np.bincount(pos // CT_T, minlength=nt) if nt else np.zeros(0, np.int64)
    rel = off - off[0]
    st = np.unique(rel[:-1])
    ts = np.arange(nt, dtype=np.int64) * CT_T
    te = np.minimum(ts + CT_T, L)
    inner = np.searchsorted(st, te, "left") - np.searchsorted(st, ts, "right")
    empty_at = rel[:-1][np.diff(rel) == 0]
    nk = len(keys)
    nt_r = -(-W // RX_T)
    npass = -(-2 * k // 8)
    digit_max, tail, runs = None, None, None
    if detail:
        digit_max, tail = [], []
        nv = nk % RX_T
        for p in range(npass):
            d = ((radix_order(keys, p) >> np.uint64(8 * p)) & np.uint64(255)).astype(np.int64)
            tile = np.arange(nk, dtype=np.int64) // RX_T
            digit_max.append(int(np.bincount(tile * RX_DIGITS + d).max()) if nk else 0)
            tail.append(bool(nv and (d[nk - nv:] == 255).any()))
        sk = np.sort(keys)
        h = np.flatnonzero(np.r_[True, sk[1:] != sk[:-1]]) if nk else np.zeros(0, np.int64)
        e = np.r_[h[1:], nk]
        runs = Runs(len(h), int(np.sum(h // SP_WB != (e - 1) // SP_WB)), int(np.sum(h // SP_WITEMS != (e - 1) // SP_WITEMS)),
                    int((e - h).max(initial=0)), int(np.sum(h % SP_WB == 0)), int(e[-1] - h[-1]) if nk else 0)
    radix = Radix(nk, nt_r, nk % RX_T, npass, bool(npass & 1), digit_max, tail, scan_passes(RX_DIGITS * nt_r))
    return Geometry(W, -(-W // CT_T), Tiles(valid, inner, empty_at), radix, runs)


def merge_geometry(table_keys, batch_keys) -> Merge:
    """The merge of a batch's distinct keys into a table: na, nb, keys in both, and whether a table key has lb = 0 or
    lb = nb (its lower bound in the batch) and a batch key has ub = 0 or ub = na (its upper bound in the table)."""
    a = np.asarray(table_keys, dtype=np.uint64)
    b = np.asarray(batch_keys, dtype=np.uint64)
    lb = np.searchsorted(b, a, "left")
    ub = np.searchsorted(a, b, "right")
    return Merge(len(a), len(b), int(np.intersect1d(a, b, assume_unique=True).size), bool((lb == 0).any()),
                 bool((lb == len(b)).any()), bool((ub == 0).any()), bool((ub == len(a)).any()))


def host_chunks(offsets):
    """(i0, i1, bases) of the host entry points' chunks: whole sequences, at most HOST_CHUNK_BASES bases each unless one
    sequence is longer (ChunkPlan in host_common.h).  A chunk with no bases is skipped by the add."""
    off = np.asarray(offsets, dtype=np.int64)
    n, cuts, i0 = len(off) - 1, [], 0
    while i0 < n:
        i1 = max(i0 + 1, min(n, int(np.searchsorted(off, off[i0] + HOST_CHUNK_BASES, "right")) - 1))
        cuts.append((i0, i1, int(off[i1] - off[i0])))
        i0 = i1
    return cuts
