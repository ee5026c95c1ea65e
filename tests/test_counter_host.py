"""Batch-wide k-mer counting (ktb_counter_*, KmerCounter, `kmertools ctr`) without a GPU: the reference table the GPU
tests compare with, argument errors of every entry point, and the CLI's parsing."""
import ctypes as C
import subprocess
from pathlib import Path

import numpy as np
import pytest

from kmertools_b200 import _lib
from oracle import oracle

from tests.util import random_batch

ROOT = Path(__file__).resolve().parent.parent
BIN = ROOT / "kmertools_b200" / "bin" / "kmertools"


def count_table(bases, offsets, k: int, canonical: bool = True):
    """(keys u64, counts u64, windows): the keys of every sequence's windows from the oracle's kmer_arrays,
    concatenated and counted with np.unique."""
    bases = np.ascontiguousarray(bases, dtype=np.uint8)
    offsets = np.asarray(offsets, dtype=np.uint64)
    keys = []
    for i in range(len(offsets) - 1):
        f, r, _ = oracle.kmer_arrays(bases[int(offsets[i]):int(offsets[i + 1])], k)
        keys.append(np.minimum(f, r) if canonical else f)
    allk = np.concatenate(keys) if keys else np.zeros(0, np.uint64)
    u, c = np.unique(allk, return_counts=True)
    return u.astype(np.uint64), c.astype(np.uint64), int(allk.size)


def pack(seqs):
    b = [s.encode() if isinstance(s, str) else s for s in seqs]
    offsets = np.zeros(len(b) + 1, dtype=np.uint64)
    np.cumsum([len(x) for x in b], out=offsets[1:])
    return np.frombuffer(b"".join(b), dtype=np.uint8), offsets


def run(*args):
    return subprocess.run([str(BIN), *map(str, args)], capture_output=True, text=True)


def test_known_answers_of_the_reference():
    """kmer/src/kmer.rs tests: canonical 2-mers of ACGT and of ACNGTT."""
    keys, counts, m = count_table(*pack(["ACGT"]), 2)
    assert dict(zip(keys.tolist(), counts.tolist())) == {1: 2, 6: 1} and m == 3
    keys, counts, m = count_table(*pack(["ACNGTT"]), 2)
    assert dict(zip(keys.tolist(), counts.tolist())) == {0: 1, 1: 2} and m == 3


@pytest.mark.parametrize("k", [1, 3, 5, 12])
def test_table_is_the_column_sum_of_the_sparse_rows(k):
    """The reference table is the sparse rows summed by code, and independent of how the batch is split."""
    from tests.sparse_ref import sparse_rows
    rng = np.random.default_rng(k)
    lens = [0, 1, k - 1, k, k + 1, 150, 600] + list(rng.integers(0, 300, size=12))
    bases, offsets = random_batch(rng, lens, noise=0.03, n_runs=0.3)
    for canonical in (True, False):
        keys, counts, m = count_table(bases, offsets, k, canonical)
        _, codes, values, totals = sparse_rows(bases, offsets, k, canonical)
        u, inv = np.unique(codes, return_inverse=True)
        want = np.zeros(len(u), np.uint64)
        np.add.at(want, inv, values.astype(np.uint64))
        assert np.array_equal(keys, u) and np.array_equal(counts, want)
        assert m == int(totals.sum()) == int(counts.sum())


def test_counter_symbols():
    for name in ("ktb_counter_create", "ktb_counter_destroy", "ktb_counter_add", "ktb_counter_add_device",
                 "ktb_counter_size", "ktb_counter_read", "ktb_counter_read_device", "ktb_count_file"):
        assert name in _lib.SYMBOLS
    from kmertools_b200 import KmerCounter  # noqa: F401
    import pykmertools
    assert not hasattr(pykmertools, "KmerCounter")


def test_counter_argument_errors():
    L = _lib.load()
    h = C.c_void_p()
    for k in (0, 32, -1):
        assert L.ktb_counter_create(k, 1, 0, C.byref(h)) == _lib.KTB_ERR_ARG
        assert b"1..31" in L.ktb_last_error()
    assert L.ktb_counter_create(21, 2, 0, C.byref(h)) == _lib.KTB_ERR_ARG
    assert b"canonical" in L.ktb_last_error()
    assert L.ktb_counter_create(21, 1, -1, C.byref(h)) == _lib.KTB_ERR_ARG
    assert L.ktb_counter_create(21, 1, 0, None) == _lib.KTB_ERR_ARG
    offs = np.array([0, 4], dtype=np.uint64)
    assert L.ktb_counter_add(None, None, offs.ctypes.data, 1) == _lib.KTB_ERR_ARG
    assert L.ktb_counter_add_device(None, None, offs.ctypes.data, 1, 4, None) == _lib.KTB_ERR_ARG
    assert L.ktb_counter_size(None, None, None) == _lib.KTB_ERR_ARG
    assert L.ktb_counter_read(None, None, None, 0) == _lib.KTB_ERR_ARG
    assert L.ktb_counter_read_device(None, None, None, 0, None) == _lib.KTB_ERR_ARG
    L.ktb_counter_destroy(None)
    assert L.ktb_count_file(None, 0, None) == _lib.KTB_ERR_ARG
    from kmertools_b200 import KmerCounter
    for k in (0, 32):
        with pytest.raises(ValueError):
            KmerCounter(k)
    if L.ktb_device_count() > 0:   # a device is visible: the device-dependent checks pass create
        assert L.ktb_counter_create(21, 1, L.ktb_device_count(), C.byref(h)) == _lib.KTB_ERR_ARG


def test_counter_without_gpu():
    L = _lib.load()
    if L.ktb_device_count() != 0:
        pytest.skip("a CUDA device is visible")
    h = C.c_void_p()
    assert L.ktb_counter_create(21, 1, 0, C.byref(h)) == _lib.KTB_ERR_NODEVICE
    assert b"no CPU path" in L.ktb_last_error()
    assert not h
    from kmertools_b200 import KmerCounter, KtbError
    with pytest.raises(KtbError):
        KmerCounter(21)


def test_ctr_cli_parsing(golden, tmp_path):
    assert BIN.exists(), "build the CLI first (python -m kmertools_b200.build)"
    fa = golden / "reads.fa"
    r = run("ctr", "-i", fa, "-k", "21")
    assert r.returncode == 2 and "--output" in r.stderr
    r = run("ctr", "-i", fa, "-o", tmp_path / "o")
    assert r.returncode == 2 and "--k-size" in r.stderr
    for k in (9, 32):
        r = run("ctr", "-i", fa, "-o", tmp_path / "o", "-k", k)
        assert r.returncode == 2 and "10..=31" in r.stderr
    r = run("ctr", "-i", fa, "-o", tmp_path / "o", "-k", "21", "--bogus")
    assert r.returncode == 2
    r = run("ctr", "-h")
    assert r.returncode == 0 and "kmers.counts" in r.stderr and "ignored" in r.stderr
    if _lib.load().ktb_device_count() == 0:
        # past parsing: the driver needs a GPU, reports it like a reference error and exits 0
        for args in (("-k", "5", "--any-k"), ("-k", "21", "-m", "8", "-a", "-t", "2")):
            r = run("ctr", "-i", fa, "-o", tmp_path / "o", *args)
            assert r.returncode == 0 and r.stderr.startswith("Error:") and "no CUDA device" in r.stderr
    else:
        r = run("ctr", "-i", fa, "-o", tmp_path / "o", "-k", "5", "--any-k")
        assert r.returncode == 0 and "10..=31" not in r.stderr
