"""Sparse (CSR) k-mer count rows without a GPU: argument checks of both entry points, the window limit of the host
entry point, and the Python restatement of the rows against the dense oracle."""
import ctypes as C

import numpy as np
import pytest

from kmertools_b200 import _lib
from oracle import oracle

from tests.sparse_ref import scatter, sparse_rows
from tests.util import random_batch


def _call_host(k=4, canonical=1, norm=0, dtype=0, offsets=None, n=None, bases=b"ACGTACGT", cap=0, codes=None,
               values=None, device=0, row_ptr=True):
    L = _lib.load()
    offs = np.array([0, len(bases)] if offsets is None else offsets, dtype=np.uint64)
    n = len(offs) - 1 if n is None else n
    buf = (C.c_uint8 * max(1, len(bases)))(*bases) if bases is not None else None
    rp = np.zeros(n + 1, dtype=np.uint64)
    return L.ktb_sparse_vectorise(buf, offs.ctypes.data, n, k, canonical, norm, dtype, device,
                                  rp.ctypes.data if row_ptr else None, codes, values, cap, None)


def test_sparse_symbols_and_limits():
    assert "ktb_sparse_vectorise" in _lib.SYMBOLS and "ktb_sparse_vectorise_device" in _lib.SYMBOLS
    from kmertools_b200 import kmer_counts, kmer_counts_tensors  # noqa: F401
    from kmertools_b200.sparse import MAX_SPARSE_K
    assert MAX_SPARSE_K == 31


def test_sparse_argument_errors():
    L = _lib.load()
    E = _lib.KTB_ERR_ARG
    for k in (0, 32, -1):
        assert _call_host(k=k) == E
        assert b"1..31" in L.ktb_last_error()
    assert _call_host(canonical=2) == E
    assert _call_host(norm=3) == E
    assert _call_host(norm=-1) == E
    assert _call_host(dtype=3) == E
    for norm in (1, 2):
        assert _call_host(norm=norm, dtype=_lib.OUT_U32) == E
        assert b"KTB_NORM_COUNTS" in L.ktb_last_error()
    assert _call_host(cap=5) == E                       # NULL codes / values with cap > 0
    assert _call_host(row_ptr=False) == E
    assert _call_host(bases=None, offsets=[0, 8]) == E  # bases NULL with bases to read
    assert _call_host(offsets=[4, 2]) == E
    assert b"non-decreasing" in L.ktb_last_error()
    # device entry point: same argument checks, before anything touches a device
    rp = np.zeros(2, dtype=np.uint64)
    offs = np.array([0, 8], dtype=np.uint64)
    dev = L.ktb_sparse_vectorise_device
    assert dev(None, offs.ctypes.data, 1, 8, 32, 1, 0, 0, rp.ctypes.data, None, None, 0, None, None) == E
    assert dev(None, offs.ctypes.data, 1, 8, 5, 1, 1, 0, rp.ctypes.data, None, None, 0, None, None) == E
    assert dev(None, offs.ctypes.data, 1, 8, 5, 1, 0, 0, rp.ctypes.data, None, None, 4, None, None) == E
    assert dev(None, offs.ctypes.data, 1, 8, 5, 1, 0, 0, None, None, None, 0, None, None) == E
    assert dev(None, offs.ctypes.data, 1, 8, 5, 1, 0, 0, rp.ctypes.data, None, None, 0, None, None) == E  # d_bases NULL
    from kmertools_b200 import kmer_counts
    with pytest.raises(ValueError):
        kmer_counts(["ACGT"], 32)
    with pytest.raises(ValueError):
        kmer_counts(["ACGT"], 0)


def test_sparse_rejects_2_pow_32_windows():
    """Counts are u32: a sequence with 2^32 windows is rejected from the offsets alone, before any base is read."""
    L = _lib.load()
    big = (1 << 32) + 30            # k = 31: exactly 2^32 windows
    assert _call_host(k=31, offsets=[0, 10, 10 + big], bases=None) == _lib.KTB_ERR_ARG
    assert b"2^32" in L.ktb_last_error() and b"sequence 1" in L.ktb_last_error()
    assert _call_host(k=1, offsets=[0, 1 << 32], bases=None) == _lib.KTB_ERR_ARG
    # one window fewer passes the limit (and then fails on the NULL bases, or on the missing device)
    rc = _call_host(k=31, offsets=[0, big - 1], bases=None)
    assert rc == _lib.KTB_ERR_ARG and b"bases is NULL" in L.ktb_last_error()


def test_sparse_without_gpu():
    L = _lib.load()
    if L.ktb_device_count() != 0:
        pytest.skip("a CUDA device is visible")
    assert _call_host() == _lib.KTB_ERR_NODEVICE
    assert b"no CPU path" in L.ktb_last_error()
    from kmertools_b200 import KtbError, kmer_counts
    with pytest.raises(KtbError):
        kmer_counts(["ACGTACGT"], 21)


@pytest.mark.parametrize("k", range(1, 9))
@pytest.mark.parametrize("canonical", [True, False])
@pytest.mark.parametrize("norm_mode", [0, 1, 2])
def test_sparse_rows_restate_the_dense_oracle(k, canonical, norm_mode):
    rng = np.random.default_rng(1000 * k + 10 * int(canonical) + norm_mode)
    lens = [0, 1, k - 1, k, k + 1, 150, 600] + list(rng.integers(0, 300, size=12))
    bases, offsets = random_batch(rng, lens, noise=0.03, n_runs=0.3)
    row_ptr, codes, values, totals = sparse_rows(bases, offsets, k, canonical, norm_mode)
    want, want_tot = oracle.vectorise_batch(bases, offsets, k, canonical, norm_mode)
    assert np.array_equal(totals, want_tot)
    assert np.all(values > 0)
    for i in range(len(lens)):
        row = codes[int(row_ptr[i]):int(row_ptr[i + 1])]
        assert np.all(np.diff(row.astype(np.int64)) > 0)
    pos_map = oracle.kmer_pos_maps(k)[0] if canonical else None
    got = scatter(row_ptr, codes, values, want.shape[1], pos_map)
    assert np.array_equal(got.view(np.uint64), want.view(np.uint64))
