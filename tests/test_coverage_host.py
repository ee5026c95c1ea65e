"""Per-read k-mer coverage histograms without a GPU: the numpy reference the GPU tests compare with, pinned against a
brute-force loop over the oracle's windows; argument errors of every entry point; the new symbols; the CLI's parsing."""
import ctypes as C
import subprocess
from pathlib import Path

import numpy as np
import pytest

from kmertools_b200 import _lib
from oracle import oracle

from tests.coverage_ref import bucket_sizes, coverage_rows, dir_bits, expected
from tests.test_counter_host import count_table
from tests.util import random_batch

ROOT = Path(__file__).resolve().parent.parent
BIN = ROOT / "kmertools_b200" / "bin" / "kmertools"


def brute_force(bases, offsets, table, k, canonical, bin_size, bin_count):
    rows, totals = [], []
    for i in range(len(offsets) - 1):
        seq = bytes(bases[int(offsets[i]):int(offsets[i + 1])])
        row = [0] * bin_count
        pairs = oracle.kmers(seq, k)
        for f, r in pairs:
            a = table.get(min(f, r) if canonical else f, 0)
            row[min(a // bin_size, bin_count - 1)] += 1
        rows.append(row)
        totals.append(len(pairs))
    return np.array(rows, np.uint64).reshape(-1, bin_count), np.array(totals, np.uint64)


@pytest.mark.parametrize("k", list(range(1, 32)))
def test_reference_equals_brute_force(k):
    rng = np.random.default_rng(300 + k)
    lens = [0, 1, k - 1, k, k + 1, 0, 200] + list(rng.integers(0, 120, size=10))
    bases, offsets = random_batch(rng, lens, noise=0.04, n_runs=0.3)
    other, other_off = random_batch(rng, list(rng.integers(0, 300, size=8)), noise=0.02)
    for canonical in (True, False):
        for src in ((bases, offsets), (other, other_off), (bases[:0], np.zeros(1, np.uint64))):
            keys, counts, _ = count_table(*src, k, canonical)
            table = dict(zip(keys.tolist(), counts.tolist()))
            for bin_size, bin_count in ((1, 1), (1, 7), (2, 5), (3, 64)):
                got = coverage_rows(bases, offsets, keys, counts, k, canonical, bin_size, bin_count)
                want = brute_force(bases, offsets, table, k, canonical, bin_size, bin_count)
                assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]), (canonical, bin_size)


def test_reference_offsets_and_large_counts():
    """offsets[0] > 0, empty records sharing a start, and counts past 2^32 binned as u64."""
    bases = np.frombuffer(b"xxACGTAAAANNAAC", np.uint8)
    offsets = np.array([2, 2, 2, 8, 8, 15], np.uint64)
    keys = np.array([0, 1, 6], np.uint64)          # AA, AC, CG at k = 2 raw
    counts = np.array([5 * 2 ** 30, 3, 1], np.uint64)
    rows, totals = coverage_rows(bases, offsets, keys, counts, 2, False, 2 ** 31, 4)
    assert totals.tolist() == [0, 0, 5, 0, 3]
    # ACGTAA: AC -> 3 (bin 0), CG -> 1, GT absent, TA absent, AA -> 5 * 2^30 (bin 2)
    assert rows[2].tolist() == [4, 0, 1, 0]
    assert rows[4].tolist() == [1, 0, 2, 0]       # AANNAAC: AA, then AA, AC
    q = expected(rows, totals, True, np.float64)
    assert q[2].tolist() == [0.8, 0.0, 0.2, 0.0] and not q[0].any()


def test_directory_rule():
    assert [dir_bits(n, 21) for n in (1, 2, 3, 4, 7, 8, 1023, 1024, 1025)] == [0, 1, 1, 2, 2, 3, 9, 10, 10]
    assert dir_bits(16, 2) == 4 and dir_bits(1000, 2) == 4      # a direct index at 2k <= b
    assert dir_bits(2 ** 40, 31) == 30
    b, sizes = bucket_sizes(np.arange(16, dtype=np.uint64), 2)
    assert b == 4 and sizes.max() == 1


def test_coverage_symbols():
    for name in ("ktb_counter_coverage", "ktb_counter_coverage_device", "ktb_coverage_file"):
        assert name in _lib.SYMBOLS
    assert _lib.load().ktb_abi_version() == 1


def test_coverage_argument_errors():
    L = _lib.load()
    offs = np.array([0, 4], dtype=np.uint64)
    out = np.zeros(16, np.float32)
    for args in ((None, None, offs.ctypes.data, 1, 16, 16, 1, 1, out.ctypes.data, None),):
        assert L.ktb_counter_coverage(*args) == _lib.KTB_ERR_ARG
    assert L.ktb_counter_coverage_device(None, None, offs.ctypes.data, 1, 4, 16, 16, 1, 1, out.ctypes.data, None,
                                         None) == _lib.KTB_ERR_ARG
    fake = C.c_void_p(1)   # never dereferenced: the NULL checks come first
    assert L.ktb_counter_coverage(fake, None, None, 1, 16, 16, 1, 1, out.ctypes.data, None) == _lib.KTB_ERR_ARG
    assert L.ktb_counter_coverage(fake, None, offs.ctypes.data, 1, 16, 16, 1, 1, None, None) == _lib.KTB_ERR_ARG
    assert L.ktb_counter_coverage_device(fake, None, None, 1, 4, 16, 16, 1, 1, out.ctypes.data, None,
                                         None) == _lib.KTB_ERR_ARG
    assert L.ktb_counter_coverage_device(fake, None, offs.ctypes.data, 1, 4, 16, 16, 1, 1, None, None,
                                         None) == _lib.KTB_ERR_ARG
    assert b"NULL" in L.ktb_last_error()


def file_opts(i, o, k=15):
    return _lib.FileOpts(str(i).encode(), str(o).encode(), k, 1, 1, b" ", 0, 0, 0)


def test_coverage_file_argument_errors(golden, tmp_path):
    L = _lib.load()
    fa = golden / "reads.fa"
    assert L.ktb_coverage_file(None, None, 16, 16, None) == _lib.KTB_ERR_ARG
    for k in (0, 32):
        assert L.ktb_coverage_file(C.byref(file_opts(fa, tmp_path / "o", k)), None, 16, 16, None) == _lib.KTB_ERR_ARG
        assert b"1..31" in L.ktb_last_error()
    o = file_opts(fa, tmp_path / "o")
    for size, count in ((0, 16), (16, 0), (16, 65537)):
        assert L.ktb_coverage_file(C.byref(o), None, size, count, None) == _lib.KTB_ERR_ARG
        assert b"bin_" in L.ktb_last_error()
    for counted in (None, b"-"):
        assert L.ktb_coverage_file(C.byref(file_opts("-", tmp_path / "o")), counted, 16, 16, None) == _lib.KTB_ERR_ARG
        assert b"read twice" in L.ktb_last_error()
    assert not (tmp_path / "o").exists()


def test_coverage_without_gpu(golden, tmp_path):
    L = _lib.load()
    if L.ktb_device_count() != 0:
        pytest.skip("a CUDA device is visible")
    from kmertools_b200 import KmerCounter, KtbError
    with pytest.raises(KtbError) as e:
        KmerCounter(15).coverage(["ACGT" * 10])
    assert e.value.code == _lib.KTB_ERR_NODEVICE
    assert L.ktb_coverage_file(C.byref(file_opts(golden / "reads.fa", tmp_path / "o")), None, 16, 16,
                               None) == _lib.KTB_ERR_NODEVICE


def cov(*args):
    return subprocess.run([str(BIN), "cov", *map(str, args)], capture_output=True, text=True)


def test_cov_cli_parsing(golden, tmp_path):
    assert BIN.exists(), "build the CLI first (python -m kmertools_b200.build)"
    fa = golden / "reads.fa"
    out = tmp_path / "o.txt"
    r = cov("-o", out)
    assert r.returncode == 2 and "--input" in r.stderr
    r = cov("-i", fa)
    assert r.returncode == 2 and "--output" in r.stderr
    for k in (9, 32):
        r = cov("-i", fa, "-o", out, "-k", k)
        assert r.returncode == 2 and "10..=31" in r.stderr
    for k in (0, 32):
        r = cov("-i", fa, "-o", out, "-k", k, "--any-k")
        assert r.returncode == 2 and "1..=31" in r.stderr
    for args in (("-i", "-"), ("-i", "-", "-a", "-")):
        r = cov(*args, "-o", out)
        assert r.returncode == 2 and "read twice" in r.stderr
    for flag, bad in (("-w", "0"), ("-w", "x"), ("-w", "4294967296"), ("-c", "0"), ("-c", "65537"), ("-c", "1.5")):
        r = cov("-i", fa, "-o", out, flag, bad)
        assert r.returncode == 2 and "invalid value" in r.stderr, (flag, bad)
    r = cov("-i", fa, "-o", out, "--bogus")
    assert r.returncode == 2
    r = cov("-h")
    assert r.returncode == 0 and "this build's own" in r.stderr and "ignored" in r.stderr
    r = subprocess.run([str(BIN), "nope"], capture_output=True, text=True)
    assert r.returncode == 2 and "kmertools cov" in r.stderr
    assert not out.exists()
    if _lib.load().ktb_device_count() == 0:
        for args in (("-k", "5", "--any-k"), ("-a", fa, "-w", "1", "-c", "65536", "-m", "8", "-t", "2")):
            r = cov("-i", fa, "-o", out, *args)
            assert r.returncode == 0 and r.stderr.startswith("Error:") and "no CUDA device" in r.stderr
