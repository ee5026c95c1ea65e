"""Sparse per-sequence k-mer counts (CSR rows) for 1 <= k <= 31 on top of ktb_sparse_vectorise*.

Row i holds the distinct keys of sequence i (canonical: min(forward, reverse complement); raw: forward) in ascending
order with their counts, normalised exactly like the dense rows of OligoComputer.  Columns are 2-bit codes
(A=0 C=1 G=2 T=3, first base most significant), as kmer_pairs returns them.
"""
from __future__ import annotations

import functools

import numpy as np

from . import _lib
from ._lib import NORM_CLI, NORM_COUNTS, OUT_F32, OUT_F64, OUT_U32
from .oligo import _CODES, _pack

MAX_SPARSE_K = 31


def _packed(seqs_or_packed):
    if isinstance(seqs_or_packed, tuple) and len(seqs_or_packed) == 2 and isinstance(seqs_or_packed[0], np.ndarray):
        bases, offsets = seqs_or_packed
        return np.ascontiguousarray(bases, dtype=np.uint8), np.ascontiguousarray(offsets, dtype=np.uint64)
    return _pack(list(seqs_or_packed))


def _check_k(ksize: int) -> int:
    if not 1 <= int(ksize) <= MAX_SPARSE_K:
        raise ValueError(f"ksize must be in 1..{MAX_SPARSE_K} (got {ksize})")
    return int(ksize)


def _check_tensors(bases, offsets, device=None):
    """Checks the CUDA tensors of a batch (uint8 bases, int64 offsets); a counter also passes the device index they must
    be on."""
    import torch
    if not (bases.is_cuda and offsets.is_cuda and bases.device == offsets.device):
        raise ValueError("bases and offsets must be CUDA tensors on one device")
    if device is not None and bases.device.index != device:
        raise ValueError(f"the tensors are on {bases.device}, the counter on cuda:{device}")
    if bases.dtype != torch.uint8 or offsets.dtype != torch.int64:
        raise TypeError(f"bases must be uint8 and offsets int64 (got {bases.dtype}, {offsets.dtype})")
    if not (bases.is_contiguous() and offsets.is_contiguous()):
        raise ValueError("bases and offsets must be contiguous")


@functools.lru_cache(maxsize=4)
def _rank_map(k: int, device: int):
    """(canonical code -> dense column as an int64 CUDA tensor of 4^k entries, number of columns), kept per (k, device):
    the table is 128 MB at k = 12."""
    import torch
    from .oligo import OligoComputer
    oc = OligoComputer(k, device=device)
    pos_map, _, dim = oc.kmer_pos_maps()
    oc.close()
    return torch.from_numpy(pos_map.astype(np.int64)).to(torch.device("cuda", device)), dim


def kmer_counts(seqs_or_packed, ksize: int, mins: bool = True, norm_mode: int = NORM_COUNTS, dtype=np.uint32,
                device: int = 0):
    """CSR rows of a batch: (row_ptr u64[n+1], codes u64[nnz], values[nnz], totals u64[n]) as numpy arrays.

    `seqs_or_packed` is a list of str / bytes, or a packed (bases u8, offsets u64[n+1]) pair as OligoComputer takes.
    dtype np.uint32 needs norm_mode NORM_COUNTS."""
    k = _check_k(ksize)
    bases, offsets = _packed(seqs_or_packed)
    n = len(offsets) - 1
    code = _CODES[np.dtype(dtype)]
    lens = np.diff(offsets.astype(np.int64)) if n else np.zeros(0, np.int64)
    cap = int(np.maximum(lens - k + 1, 0).sum())
    row_ptr = np.zeros(n + 1, dtype=np.uint64)
    codes = np.empty(cap, dtype=np.uint64)
    values = np.empty(cap, dtype=np.dtype(dtype))
    totals = np.zeros(n, dtype=np.uint64)
    _lib.check(_lib.load().ktb_sparse_vectorise(
        bases.ctypes.data if bases.size else None, offsets.ctypes.data, n, k, int(mins), int(norm_mode), code,
        int(device), row_ptr.ctypes.data, codes.ctypes.data if cap else None, values.ctypes.data if cap else None,
        cap, totals.ctypes.data if n else None))
    nnz = int(row_ptr[-1])
    if nnz < cap:
        codes, values = codes[:nnz].copy(), values[:nnz].copy()
    return row_ptr, codes, values, totals


def kmer_counts_tensors(bases, offsets, ksize: int, mins: bool = True, norm_mode: int = NORM_CLI, dtype=None,
                        columns: str = "code"):
    """CSR rows of CUDA tensors as a torch.sparse_csr_tensor of size (n, 4**ksize), computed on torch's current stream.

    `bases` (uint8) and `offsets` (int64, n+1, absolute positions in `bases`) live on one GPU.  columns="rank" (canonical
    rows with ksize <= 12 only) numbers the columns like OligoComputer's dense rows, size (n, dim), so `.to_dense()`
    equals OligoComputer.vectorise_tensors.  The call reads row_ptr[n] back to the host once (it waits for the stream)
    to size the result; codes and values are views of buffers sized for every window of the batch.

    Scratch and outputs are sized from bases.numel(), not from the span of the offsets: for a small batch inside a large
    buffer, pass the slice bases[offsets[0]:offsets[n]] and offsets - offsets[0]."""
    import torch
    k = _check_k(ksize)
    _check_tensors(bases, offsets)
    if columns not in ("code", "rank"):
        raise ValueError(f"columns must be 'code' or 'rank' (got {columns!r})")
    if columns == "rank" and (not mins or k > _lib.MAX_K):
        raise ValueError(f"columns='rank' needs canonical rows and ksize <= {_lib.MAX_K}")
    dtype = dtype or torch.float32
    codes_of = {torch.int32: OUT_U32, torch.float32: OUT_F32, torch.float64: OUT_F64}
    if dtype not in codes_of:
        raise TypeError(f"dtype must be torch.int32, torch.float32 or torch.float64 (got {dtype})")
    code = codes_of[dtype]
    n = offsets.numel() - 1
    dev = bases.device
    total = bases.numel()   # a bound of offsets[n]; sizes the scratch and the outputs
    cap = max(total, 1)
    row_ptr = torch.empty(n + 1, dtype=torch.int64, device=dev)
    codes = torch.empty(cap, dtype=torch.int64, device=dev)
    values = torch.empty(cap, dtype=dtype, device=dev)
    with torch.cuda.device(dev):
        stream = torch.cuda.current_stream(dev).cuda_stream
        _lib.check(_lib.load().ktb_sparse_vectorise_device(
            bases.data_ptr() if total else None, offsets.data_ptr(), n, total, k, int(mins), int(norm_mode), code,
            row_ptr.data_ptr(), codes.data_ptr(), values.data_ptr(), cap, None, stream))
    nnz = int(row_ptr[-1])
    cols = codes[:nnz]
    if columns == "rank":
        pos_map, dim = _rank_map(k, dev.index)
        cols = pos_map[cols]
        size = (n, dim)
    else:
        size = (n, 4 ** k)
    return torch.sparse_csr_tensor(row_ptr, cols, values[:nnz], size=size)
