"""Python restatement of the sparse rows (ktb_sparse_vectorise*): the windows of each sequence from the oracle's
kmer_arrays, their keys counted with np.unique, and the dense rows' normalisation.  Slow; for tests."""
from __future__ import annotations

import numpy as np

from oracle import oracle

NORM_COUNTS, NORM_CLI, NORM_PY = 0, 1, 2


def sparse_rows(bases: np.ndarray, offsets: np.ndarray, k: int, canonical: bool = True, norm_mode: int = NORM_COUNTS):
    """(row_ptr u64[n+1], codes u64[nnz], values f64[nnz], totals u64[n]); values in f64 (counts when NORM_COUNTS).

    The f32 row is values.astype(np.float32) and the u32 row values.astype(np.uint32), as for the dense oracle."""
    bases = np.ascontiguousarray(bases, dtype=np.uint8)
    offsets = np.asarray(offsets, dtype=np.uint64)
    n = len(offsets) - 1
    row_ptr = np.zeros(n + 1, dtype=np.uint64)
    totals = np.zeros(n, dtype=np.uint64)
    codes, values = [], []
    for i in range(n):
        f, r, m = oracle.kmer_arrays(bases[int(offsets[i]):int(offsets[i + 1])], k)
        keys = np.minimum(f, r) if canonical else f
        u, c = np.unique(keys, return_counts=True)
        totals[i] = m
        div = max(1, 2 * m if (norm_mode == NORM_PY and not canonical) else m)
        v = c.astype(np.float64)
        if norm_mode != NORM_COUNTS:
            v = v / np.float64(div)
        codes.append(u.astype(np.uint64))
        values.append(v)
        row_ptr[i + 1] = row_ptr[i] + len(u)
    cat = (lambda xs, dt: np.concatenate(xs).astype(dt) if xs else np.zeros(0, dt))
    return row_ptr, cat(codes, np.uint64), cat(values, np.float64), totals


def scatter(row_ptr: np.ndarray, codes: np.ndarray, values: np.ndarray, dim: int, pos_map: np.ndarray | None = None,
            dtype=np.float64) -> np.ndarray:
    """Dense n x dim rows from CSR rows; columns through pos_map (canonical) or the codes themselves (raw)."""
    n = len(row_ptr) - 1
    out = np.zeros((n, dim), dtype=dtype)
    rows = np.repeat(np.arange(n), np.diff(row_ptr.astype(np.int64)))
    cols = pos_map[codes].astype(np.int64) if pos_map is not None else codes.astype(np.int64)
    out[rows, cols] = values
    return out
