"""Reference of the per-read k-mer coverage histograms (ktb_counter_coverage*, KmerCounter.coverage, `kmertools cov`)
and a Python restatement of the lookup directory the GPU builds over the counter's table (csrc/counter.cu)."""
from __future__ import annotations

import numpy as np

from tests.counter_geometry import position_keys

MAX_DIR_BITS = 30            # COV_MAX_DIR_BITS (coverage_kernels.cuh)


def coverage_rows(bases, offsets, table_keys, table_counts, k: int, canonical: bool, bin_size: int, bin_count: int):
    """(rows u64 (n, bin_count), totals u64 (n,)): per sequence, the histogram of min(a // bin_size, bin_count - 1) over
    its valid windows, a = the count of the window's key in the table (0 when absent)."""
    off = np.asarray(offsets, dtype=np.int64)
    n = len(off) - 1
    pos, keys = position_keys(bases, off, k, canonical)
    tk = np.asarray(table_keys, dtype=np.uint64)
    tc = np.asarray(table_counts, dtype=np.uint64)
    a = np.zeros(len(keys), np.uint64)
    if len(tk):
        at = np.searchsorted(tk, keys)
        found = at < len(tk)
        found[found] = tk[at[found]] == keys[found]
        a[found] = tc[at[found]]
    b = np.minimum(a // np.uint64(bin_size), np.uint64(bin_count - 1)).astype(np.int64)
    seq = np.searchsorted(off - off[0], pos, "right") - 1          # the last sequence starting at or before pos
    rows = np.bincount(seq * bin_count + b, minlength=n * bin_count).astype(np.uint64).reshape(n, bin_count)
    return rows, rows.sum(axis=1, dtype=np.uint64)


def expected(rows, totals, norm: bool, dtype):
    """The rows as the library returns them: u32 counts, or count / max(1, total) as the f64 quotient (f32: rounded
    once from it)."""
    dtype = np.dtype(dtype)
    if not norm:
        return rows.astype(dtype)
    q = rows.astype(np.float64) / np.maximum(totals, 1).astype(np.float64)[:, None]
    return q.astype(dtype)


def dir_bits(nkeys: int, k: int) -> int:
    """b of the directory over a table of nkeys keys: floor(log2 nkeys), capped at 2k and at MAX_DIR_BITS."""
    return min(max(nkeys, 1).bit_length() - 1, 2 * k, MAX_DIR_BITS)


def bucket_sizes(table_keys, k: int):
    """(b, keys per bucket of the directory) for a non-empty table."""
    keys = np.asarray(table_keys, dtype=np.uint64)
    b = dir_bits(len(keys), k)
    return b, np.bincount((keys >> np.uint64(2 * k - b)).astype(np.int64), minlength=1 << b)
