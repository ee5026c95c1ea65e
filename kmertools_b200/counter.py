"""Batch-wide k-mer counting for 1 <= k <= 31 on top of ktb_counter_* (the table of `kmertools ctr`).

A KmerCounter keeps one table on its GPU: every distinct key seen so far (canonical: min(forward, reverse complement);
raw: forward) in ascending order, with a u64 count of its windows.  Keys are 2-bit codes (A=0 C=1 G=2 T=3, first base
most significant), as kmer_pairs and kmer_counts return them.  The table does not depend on how the input is split
into adds or on their order.

coverage / coverage_tensors look every window of a batch up in that table and return per-sequence histograms of the
abundances (this build's own semantics, include/kmertools_b200.h): bin min(a // bin_size, bin_count - 1) of a window
whose key has count a (0 when absent), rows normalised by the sequence's valid windows or as u32 counts.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from .oligo import _CODES
from .sparse import _check_k, _check_tensors, _packed


class KmerCounter:
    """KmerCounter(ksize, mins=True, device=0): add batches with add / add_tensors, read the table with result /
    result_tensors.  Every add returns when the batch is in the table."""

    def __init__(self, ksize: int, mins: bool = True, device: int = 0):
        self.ksize = _check_k(ksize)
        self.mins = bool(mins)
        self.device = int(device)
        self._h = C.c_void_p()
        self._read = None   # CUDA event after the copies of the last result_tensors: the next add waits for it
        _lib.check(_lib.load().ktb_counter_create(self.ksize, int(self.mins), self.device, C.byref(self._h)))

    def _handle(self):
        if not self._h:
            raise ValueError("the counter is closed")
        return self._h

    def add(self, seqs_or_packed) -> None:
        """Counts a list of str / bytes, or a packed (bases u8, offsets u64[n+1]) pair, from host memory.  Waits on the
        host for the copies of an earlier result_tensors, which read the table this add replaces."""
        bases, offsets = _packed(seqs_or_packed)
        n = len(offsets) - 1
        if self._read is not None:
            self._read.synchronize()
            self._read = None
        _lib.check(_lib.load().ktb_counter_add(self._handle(), bases.ctypes.data if bases.size else None,
                                               offsets.ctypes.data, max(n, 0)))

    def add_tensors(self, bases, offsets) -> None:
        """Counts CUDA tensors on the counter's device, on torch's current stream: `bases` uint8, `offsets` int64 (n+1,
        absolute positions in `bases`).  The scratch is sized from bases.numel(): for a small batch inside a large
        buffer, pass the slice bases[offsets[0]:offsets[n]] and offsets - offsets[0].  The current stream first waits
        for the copies of an earlier result_tensors, which read the table this add replaces."""
        import torch
        _check_tensors(bases, offsets, self.device)
        n = offsets.numel() - 1
        total = bases.numel()
        with torch.cuda.device(bases.device):
            current = torch.cuda.current_stream(bases.device)
            if self._read is not None:
                current.wait_event(self._read)
            stream = current.cuda_stream
            _lib.check(_lib.load().ktb_counter_add_device(self._handle(), bases.data_ptr() if total else None,
                                                          offsets.data_ptr(), max(n, 0), total, stream))

    def _size(self):
        nkeys, nwin = C.c_uint64(), C.c_uint64()
        _lib.check(_lib.load().ktb_counter_size(self._handle(), C.byref(nkeys), C.byref(nwin)))
        return nkeys.value, nwin.value

    def __len__(self) -> int:
        return self._size()[0]

    @property
    def windows(self) -> int:
        """Valid windows added so far (the sum of the counts)."""
        return self._size()[1]

    def result(self):
        """(keys u64, counts u64) as numpy arrays, keys ascending."""
        n = len(self)
        keys = np.empty(n, dtype=np.uint64)
        counts = np.empty(n, dtype=np.uint64)
        _lib.check(_lib.load().ktb_counter_read(self._handle(), keys.ctypes.data if n else None,
                                                counts.ctypes.data if n else None, n))
        return keys, counts

    def result_tensors(self):
        """(keys, counts) as int64 CUDA tensors on the counter's device, copied on torch's current stream.  The copies
        read the table in place; the next add or add_tensors waits for them, so the tensors hold this table."""
        import torch
        n = len(self)
        dev = torch.device("cuda", self.device)
        keys = torch.empty(n, dtype=torch.int64, device=dev)
        counts = torch.empty(n, dtype=torch.int64, device=dev)
        with torch.cuda.device(dev):
            stream = torch.cuda.current_stream(dev).cuda_stream
            _lib.check(_lib.load().ktb_counter_read_device(self._handle(), keys.data_ptr() if n else None,
                                                           counts.data_ptr() if n else None, n, stream))
            if n:
                self._read = torch.cuda.Event()
                self._read.record()
        return keys, counts

    def _coverage_args(self, bin_size, bin_count, norm, dtype, torch_dtypes=None):
        bin_size, bin_count = int(bin_size), int(bin_count)
        if not 1 <= bin_size < 2 ** 32:
            raise ValueError(f"bin_size must be in 1..2^32-1 (got {bin_size})")
        if not 1 <= bin_count <= 65536:
            raise ValueError(f"bin_count must be in 1..65536 (got {bin_count})")
        codes = torch_dtypes or _CODES
        key = dtype if torch_dtypes else np.dtype(dtype)
        if key not in codes:
            raise TypeError(f"dtype must be uint32, float32 or float64 (got {dtype})")
        out = codes[key]
        if out == _lib.OUT_U32 and norm:
            raise ValueError("uint32 rows are counts: pass norm=False")
        return bin_size, bin_count, (_lib.NORM_CLI if norm else _lib.NORM_COUNTS), out

    def coverage(self, seqs_or_packed, bin_size: int = 16, bin_count: int = 16, norm: bool = True, dtype=np.float32):
        """Coverage histograms of a list of str / bytes, or a packed (bases u8, offsets u64[n+1]) pair, from host
        memory: (rows (n, bin_count) of dtype, totals u64 (n,)).  Synchronous; reads the table in place."""
        bin_size, bin_count, norm_mode, out = self._coverage_args(bin_size, bin_count, norm, dtype)
        bases, offsets = _packed(seqs_or_packed)
        n = max(len(offsets) - 1, 0)
        rows = np.zeros((n, bin_count), dtype=np.dtype(dtype))
        totals = np.zeros(n, dtype=np.uint64)
        _lib.check(_lib.load().ktb_counter_coverage(self._handle(), bases.ctypes.data if bases.size else None,
                                                    offsets.ctypes.data, n, bin_size, bin_count, norm_mode, out,
                                                    rows.ctypes.data, totals.ctypes.data))
        return rows, totals

    def coverage_tensors(self, bases, offsets, bin_size: int = 16, bin_count: int = 16, norm: bool = True, dtype=None):
        """coverage of CUDA tensors (the arguments of add_tensors) on torch's current stream: (rows (n, bin_count),
        totals int64 (n,)) as CUDA tensors; dtype torch.float32 (default), torch.float64 or torch.int32 (u32 counts,
        norm=False).  The kernels read the table in place; the next add or add_tensors waits for them."""
        import torch
        if dtype is None:
            dtype = torch.float32
        bin_size, bin_count, norm_mode, out = self._coverage_args(
            bin_size, bin_count, norm, dtype,
            {torch.int32: _lib.OUT_U32, torch.float32: _lib.OUT_F32, torch.float64: _lib.OUT_F64})
        _check_tensors(bases, offsets, self.device)
        n = max(offsets.numel() - 1, 0)
        total = bases.numel()
        rows = torch.empty((n, bin_count), dtype=dtype, device=bases.device)
        totals = torch.empty(n, dtype=torch.int64, device=bases.device)
        with torch.cuda.device(bases.device):
            current = torch.cuda.current_stream(bases.device)
            _lib.check(_lib.load().ktb_counter_coverage_device(
                self._handle(), bases.data_ptr() if total else None, offsets.data_ptr(), n, total, bin_size,
                bin_count, norm_mode, out, rows.data_ptr() if n else None, totals.data_ptr() if n else None,
                current.cuda_stream))
            if n:
                self._read = torch.cuda.Event()
                self._read.record(current)
        return rows, totals

    def close(self) -> None:
        if self._h:
            _lib.load().ktb_counter_destroy(self._h)
            self._h = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
