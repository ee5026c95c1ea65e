"""Per-read k-mer coverage histograms on the GPU (ktb_counter_coverage*, KmerCounter.coverage, `kmertools cov`).  Every
case compares rows (bit for bit: u32 counts, f32 and f64 quotients) and totals with tests/coverage_ref.py."""
import subprocess
import threading
from pathlib import Path

import numpy as np
import pytest

from kmertools_b200 import KmerCounter, _lib
from kmertools_b200.io import read_fastx
from oracle import oracle

from tests.coverage_ref import bucket_sizes, coverage_rows, dir_bits, expected
from tests.counter_geometry import CT_T, host_chunks
from tests.test_counter_host import pack
from tests.util import random_batch

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

ROOT = Path(__file__).resolve().parent.parent
BIN = ROOT / "kmertools_b200" / "bin" / "kmertools"
DEV = torch.device("cuda", 0)
PARITY_K = [1, 2, 5, 10, 12, 13, 15, 16, 21, 28, 31]
BINS = [(1, 1), (1, 7), (16, 16), (3, 65536), (2 ** 31, 4)]
MODES = [(False, np.uint32, torch.int32), (True, np.float32, torch.float32), (True, np.float64, torch.float64)]


def on_device(bases, offsets):
    return torch.from_numpy(np.array(bases)).to(DEV), torch.from_numpy(offsets.astype(np.int64)).to(DEV)


def as_np(t, npdt):
    a = t.cpu().numpy()
    return a.view(np.uint32) if npdt == np.uint32 else a


def check(c, bases, offsets, bin_size, bin_count, host=True, device=True, what=""):
    """Rows and totals of both entry points in every (norm, dtype) against the reference over c's table."""
    keys, counts = c.result()
    rows, totals = coverage_rows(bases, offsets, keys, counts, c.ksize, c.mins, bin_size, bin_count)
    for norm, npdt, tdt in MODES:
        want = expected(rows, totals, norm, npdt)
        if host:
            got, tot = c.coverage((bases, offsets), bin_size, bin_count, norm, npdt)
            assert got.dtype == npdt and np.array_equal(got, want), f"{what} host {npdt}"
            assert np.array_equal(tot, totals), what
        if device:
            got, tot = c.coverage_tensors(*on_device(bases, offsets), bin_size, bin_count, norm, tdt)
            assert np.array_equal(as_np(got, npdt), want), f"{what} device {npdt}"
            assert np.array_equal(tot.cpu().numpy().astype(np.uint64), totals), what
    return rows, totals


def table_state(c):
    keys, counts = c.result()
    return keys, counts, len(c), c.windows


# ---------------------------------------------------------------------------------------------------- arguments
def test_argument_errors_leave_the_counter():
    rng = np.random.default_rng(1)
    bases, offsets = random_batch(rng, [300, 50, 0, 900])
    tb, to = on_device(bases, offsets)
    L = _lib.load()
    out = torch.zeros(4 * 65537, dtype=torch.float64, device=DEV)
    with KmerCounter(13) as c:
        c.add((bases, offsets))
        before = table_state(c)
        for bs, bc, norm, dt in ((0, 16, 1, 1), (16, 0, 1, 1), (16, 65537, 1, 1), (16, 16, _lib.NORM_PY, 1),
                                 (16, 16, 1, _lib.OUT_U32), (16, 16, 0, 3), (16, 16, 3, 1)):
            rc = L.ktb_counter_coverage_device(c._h, tb.data_ptr(), to.data_ptr(), 4, tb.numel(), bs, bc, norm, dt,
                                               out.data_ptr(), None, None)
            assert rc == _lib.KTB_ERR_ARG, (bs, bc, norm, dt)
            host = np.zeros(4 * 65537, np.float64)
            rc = L.ktb_counter_coverage(c._h, bases.ctypes.data, offsets.ctypes.data, 4, bs, bc, norm, dt,
                                        host.ctypes.data, None)
            assert rc == _lib.KTB_ERR_ARG and not host.any()
        after = table_state(c)
        assert all(np.array_equal(x, y) for x, y in zip(before[:2], after[:2])) and before[2:] == after[2:]
        with pytest.raises(ValueError):
            c.coverage((bases, offsets), dtype=np.uint32)        # u32 rows are counts
        with pytest.raises(ValueError):
            c.coverage((bases, offsets), bin_count=65537)
        check(c, bases, offsets, 16, 16, what="after the errors")


# ------------------------------------------------------------------------------------------------------- parity
@pytest.mark.parametrize("k", PARITY_K)
@pytest.mark.parametrize("canonical", [True, False])
def test_parity(k, canonical):
    rng = np.random.default_rng(1000 * k + int(canonical))
    lens = [0, 1, k - 1, k, k + 1, 0, 4095, 4096, 4097, 3 * 4096 + 17] + list(rng.integers(0, 400, size=30))
    bases, offsets = random_batch(rng, lens, noise=0.03, n_runs=0.3)
    # repeats so that abundances spread over several bins
    bases[int(offsets[12]):int(offsets[13])] = np.resize(bases[int(offsets[11]):int(offsets[12])], int(offsets[13] - offsets[12]))
    other = random_batch(rng, list(rng.integers(0, 2000, size=20)), noise=0.01)
    with KmerCounter(k, canonical) as same, KmerCounter(k, canonical) as diff:
        same.add((bases, offsets))
        same.add((bases[:int(offsets[20])], offsets[:21]))
        diff.add(other)
        diff.add((bases[:int(offsets[8])], offsets[:9]))
        for bin_size, bin_count in BINS:
            nb = 8 if bin_count == 65536 else len(lens)       # keep the 65536-bin rows small
            sb, so = bases[:int(offsets[nb])], offsets[:nb + 1]
            check(same, sb, so, bin_size, bin_count, what=f"same {bin_size}x{bin_count}")
            check(diff, sb, so, bin_size, bin_count, what=f"other {bin_size}x{bin_count}")


# ------------------------------------------------------------------------------------------------ directory shapes
def distinct_kmer_batch(rng, k, nkeys, canonical=False):
    """nkeys records of length k holding nkeys distinct k-mers (raw keys), their repeats at random."""
    codes = rng.choice(4 ** k, size=nkeys, replace=False) if k <= 12 else np.unique(rng.integers(0, 4 ** k, size=nkeys + 64, dtype=np.uint64))[:nkeys]
    seqs = [oracle.numeric_to_kmer(int(x), k).encode() for x in codes]
    return pack(seqs * 2)


def test_empty_counter():
    rng = np.random.default_rng(2)
    bases, offsets = random_batch(rng, [0, 5, 400, 4100], noise=0.02)
    for k in (1, 21, 31):
        with KmerCounter(k) as c:
            rows, totals = check(c, bases, offsets, 1, 5, what=f"empty k={k}")
            assert np.array_equal(rows[:, 0], totals) and not rows[:, 1:].any()


@pytest.mark.parametrize("nkeys", [1, 2, 3, 4, 7, 8, 9, 1023, 1024, 1025, 65535, 65536, 65537])
def test_directory_sizes(nkeys):
    rng = np.random.default_rng(nkeys)
    k = 12
    bases, offsets = distinct_kmer_batch(rng, k, nkeys)
    query = np.concatenate([bases, random_batch(rng, [3000])[0]])
    qoff = np.concatenate([offsets, [offsets[-1] + 3000]]).astype(np.uint64)
    with KmerCounter(k, False) as c:
        c.add((bases, offsets))
        keys, _ = c.result()
        assert len(keys) == nkeys
        b, sizes = bucket_sizes(keys, k)
        assert b == dir_bits(nkeys, k) == nkeys.bit_length() - 1 and sizes.max() <= 2 ** (2 * k - b)
        check(c, query, qoff, 1, 4, host=nkeys < 100, what=f"nkeys={nkeys}")


@pytest.mark.parametrize("k", [1, 2, 5])
def test_direct_index(k):
    """Every raw k-mer in the table: b = 2k, one key per bucket."""
    seqs = [oracle.numeric_to_kmer(x, k).encode() * (1 + x % 3) for x in range(4 ** k)]
    bases, offsets = pack(seqs)
    with KmerCounter(k, False) as c:
        c.add((bases, offsets))
        keys, _ = c.result()
        b, sizes = bucket_sizes(keys, k)
        assert b == 2 * k and sizes.max() == 1
        check(c, bases, offsets, 2, 9, what=f"direct k={k}")


def test_one_full_bucket():
    """256 keys that differ only in their last 4 bases: at k = 31, b = 8 and every key has the same top 8 bits."""
    rng = np.random.default_rng(4)
    stem = bytes(rng.choice(list(b"ACGT"), size=27).astype(np.uint8))
    seqs = [stem + oracle.numeric_to_kmer(x, 4).encode() for x in range(256)]
    bases, offsets = pack(seqs + seqs[:100])
    with KmerCounter(31, False) as c:
        c.add((bases, offsets))
        keys, _ = c.result()
        b, sizes = bucket_sizes(keys, 31)
        assert len(keys) == 256 and b == 8 and sizes.max() == 256
        query = np.concatenate([bases, random_batch(rng, [500])[0]])
        check(c, query, np.append(offsets, offsets[-1] + 500).astype(np.uint64), 1, 3, what="full bucket")


@pytest.mark.parametrize("k", [7, 31])
def test_extreme_keys(k):
    """Keys 0 (poly-A) and 4^k - 1 (poly-T) in raw mode: the first and the last bucket; at k = 31 with two or three
    keys the prefix is bits 61 and up."""
    for extra in ([], [b"ACGT" * 10]):
        bases, offsets = pack([b"A" * (k + 3), b"T" * (k + 1)] + extra)
        with KmerCounter(k, False) as c:
            c.add((bases, offsets))
            keys, _ = c.result()
            assert keys[0] == 0 and keys[-1] == 4 ** k - 1
            b, _ = bucket_sizes(keys, k)
            assert 2 * k - b >= (61 if k == 31 and not extra else 0)
            q, qo = pack([b"A" * 50, b"T" * 50, b"ACGT" * 20, b"G" * 40])
            check(c, q, qo, 1, 6, what=f"extremes k={k}")


@pytest.mark.parametrize("k", [1, 31])
def test_abundance_past_2_pow_32(k):
    n = 1 << 30
    tb = torch.full((n,), ord("A"), dtype=torch.uint8, device=DEV)
    to = torch.tensor([0, n], dtype=torch.int64, device=DEV)
    with KmerCounter(k) as c:
        for _ in range(5):
            c.add_tensors(tb, to)
        del tb
        a = 5 * (n - k + 1)
        assert a > 2 ** 32 and a // 2 ** 31 == 2
        bases, offsets = pack([b"A" * 40, b"C" * 40, b"AG" * 40])
        rows, _ = check(c, bases, offsets, 2 ** 31, 4, what=f"u64 abundance k={k}")
        assert rows[0].tolist() == [0, 0, 40 - k + 1, 0]
    torch.cuda.empty_cache()


# ------------------------------------------------------------------------------------------------- batch shapes
def test_tile_edges_and_empty_records():
    rng = np.random.default_rng(5)
    lens = [CT_T - 1, 1, CT_T, 0, 0, CT_T + 1, 5, 2 * CT_T - 3, 0] + [7] * 600 + [CT_T * 3]
    bases, offsets = random_batch(rng, lens, noise=0.01)
    nrec = np.frombuffer(b"N" * 300, np.uint8)
    bases = np.concatenate([bases, nrec])
    offsets = np.append(offsets, offsets[-1] + 300).astype(np.uint64)
    with KmerCounter(11) as c:
        c.add((bases, offsets))
        rows, totals = check(c, bases, offsets, 2, 8, what="tile edges")
    assert totals[3] == totals[4] == totals[-1] == 0 and totals[1] == 0 and not rows[[1, 3, 4, -1]].any()


def test_long_record_f32_divisor():
    """A 2^24 + 3 base record: the divisor is >= 2^24, past the exact f32 reciprocal path."""
    rng = np.random.default_rng(6)
    bases, offsets = random_batch(rng, [(1 << 24) + 3, 100])
    with KmerCounter(3) as c:
        c.add((bases, offsets))
        _, totals = check(c, bases, offsets, 50_000, 16, what="2^24 + 3")
        assert totals[0] >= 1 << 24


@pytest.fixture(scope="module")
def reads_1m():
    import bench
    return bench.make_workload_torch(bench.WORKLOADS["reads150_k5"], 0.1, DEV)


def test_a_million_reads(reads_1m):
    tb, to = reads_1m
    assert to.numel() - 1 == 1_000_000
    bases, offsets = tb.cpu().numpy(), to.cpu().numpy().astype(np.uint64)
    with KmerCounter(11) as c:   # a table of at most 2^21 keys keeps the reference's searchsorted short
        c.add_tensors(tb, to)
        check(c, bases, offsets, 8, 16, host=False, what="10^6 reads")


def sparse_codes_values(tb, to, k, mins):
    n, total = to.numel() - 1, tb.numel()
    row_ptr = torch.empty(n + 1, dtype=torch.int64, device=DEV)
    codes = torch.empty(total, dtype=torch.int64, device=DEV)
    values = torch.empty(total, dtype=torch.int32, device=DEV)
    _lib.check(_lib.load().ktb_sparse_vectorise_device(
        tb.data_ptr(), to.data_ptr(), n, total, k, int(mins), _lib.NORM_COUNTS, _lib.OUT_U32, row_ptr.data_ptr(),
        codes.data_ptr(), values.data_ptr(), total, None, torch.cuda.current_stream(DEV).cuda_stream))
    nnz = int(row_ptr[-1])
    return row_ptr, codes[:nnz], values[:nnz]


def test_cross_check_with_the_sparse_rows(reads_1m):
    """Each read's sparse row (distinct codes and their counts), joined with the table by searchsorted and binned with
    torch, equals the coverage rows: a check that does not go through the reference."""
    tb, to = reads_1m
    k, bin_size, bin_count = 21, 1, 8
    n = to.numel() - 1
    other = torch.cat([tb[: 75_000_000], tb[: 10_000_000]])
    with KmerCounter(k) as c:
        c.add_tensors(other, torch.tensor([0, 70_000_000, other.numel()], dtype=torch.int64, device=DEV))
        keys, counts = c.result_tensors()
        rows, totals = c.coverage_tensors(tb, to, bin_size, bin_count, norm=False, dtype=torch.int32)
        row_ptr, codes, values = sparse_codes_values(tb, to, k, True)
        at = torch.searchsorted(keys, codes).clamp_(max=max(len(keys) - 1, 0))
        a = torch.where(keys[at] == codes, counts[at], torch.zeros_like(codes))
        b = torch.clamp(a // bin_size, max=bin_count - 1)
        seq = torch.repeat_interleave(torch.arange(n, device=DEV), row_ptr[1:] - row_ptr[:-1])
        want = torch.zeros(n * bin_count, dtype=torch.int64, device=DEV)
        want.scatter_add_(0, seq * bin_count + b, values.to(torch.int64))
        assert torch.equal(rows.to(torch.int64).view(-1), want)
        assert torch.equal(totals, want.view(n, bin_count).sum(1))
        assert int((want.view(n, bin_count)[:, 0]).sum()) > 0 and int(want.view(n, bin_count)[:, 1:].sum()) > 0


def test_device_entry_offsets_fences_and_streams():
    rng = np.random.default_rng(9)
    bases, offsets = random_batch(rng, list(rng.integers(0, 600, size=300)) + [0, 9000], noise=0.02)
    n, bc = len(offsets) - 1, 5
    pad = np.frombuffer(b"ACGT" * 2500, np.uint8)
    L = _lib.load()
    with KmerCounter(17) as c:
        c.add((bases, offsets))
        keys, counts = c.result()
        rows, totals = coverage_rows(bases, offsets, keys, counts, 17, True, 1, bc)
        tb, to = on_device(np.concatenate([pad, bases, pad]), offsets + len(pad))
        for norm, npdt, tdt in MODES:
            esz = np.dtype(npdt).itemsize
            g = 64 // esz
            fence = torch.full((n * bc + 2 * g,), 7, dtype=tdt, device=DEV)
            tfence = torch.full((n + 16,), -3, dtype=torch.int64, device=DEV)
            _lib.check(L.ktb_counter_coverage_device(
                c._h, tb.data_ptr(), to.data_ptr(), n, tb.numel(), 1, bc, int(norm), {np.uint32: 0, np.float32: 1,
                np.float64: 2}[npdt], fence.data_ptr() + 64, tfence.data_ptr() + 64, None))
            torch.cuda.synchronize()
            got = fence[g:g + n * bc].view(n, bc)
            assert np.array_equal(as_np(got, npdt), expected(rows, totals, norm, npdt))
            assert bool((fence[:g] == 7).all()) and bool((fence[g + n * bc:] == 7).all())
            assert np.array_equal(tfence[8:8 + n].cpu().numpy().astype(np.uint64), totals)
            assert bool((tfence[:8] == -3).all()) and bool((tfence[8 + n:] == -3).all())
        # two batches on two streams at once, the same counter read by both
        other = random_batch(rng, list(rng.integers(0, 5000, size=200)))
        batches = [on_device(bases, offsets), on_device(*other)]
        wants = [rows, coverage_rows(*other, keys, counts, 17, True, 1, bc)[0]]
        streams = [torch.cuda.Stream(DEV), torch.cuda.Stream(DEV)]
        results = [None, None]

        def work(i):
            with torch.cuda.stream(streams[i]):
                for _ in range(3):
                    results[i] = c.coverage_tensors(*batches[i], 1, bc, norm=False, dtype=torch.int32)[0]
                streams[i].synchronize()

        threads = [threading.Thread(target=work, args=(i,)) for i in range(2)]
        for t in threads:
            t.start()
        for t in threads:
            t.join()
        for r, w in zip(results, wants):
            assert np.array_equal(as_np(r, np.uint32), w.astype(np.uint32))


def test_host_chunks_equal_the_device_entry():
    rng = np.random.default_rng(10)
    lens = [150] * 300_000 + [70_000_000] + list(rng.integers(0, 1000, size=100_000)) + [0, 7]
    bases, offsets = random_batch(rng, lens, noise=0.001, n_runs=0.01)
    assert len(host_chunks(offsets)) >= 3
    with KmerCounter(19) as c:
        c.add((bases[:20_000_000], offsets[offsets <= 20_000_000]))
        h, ht = c.coverage((bases, offsets), 1, 8, False, np.uint32)
        d, dt = c.coverage_tensors(*on_device(bases, offsets), 1, 8, False, torch.int32)
        assert np.array_equal(h, as_np(d, np.uint32)) and np.array_equal(ht, dt.cpu().numpy().astype(np.uint64))
        keys, counts = c.result()
        sub = 300_000
        want = coverage_rows(bases[:int(offsets[sub])], offsets[:sub + 1], keys, counts, 19, True, 1, 8)[0]
        assert np.array_equal(h[:sub], want.astype(np.uint32))


# ------------------------------------------------------------------------------------------------------ ordering
def test_ordering_against_adds():
    rng = np.random.default_rng(11)
    bases, offsets = random_batch(rng, list(rng.integers(100, 3000, size=200)))
    other = random_batch(rng, list(rng.integers(100, 3000, size=200)))
    tb, to = on_device(bases, offsets)
    with KmerCounter(13) as c:
        c.add(other)
        first = c.coverage((bases, offsets), 1, 4, False, np.uint32)
        c.coverage_tensors(tb, to, 1, 4)
        ev = c._read
        c.add((bases, offsets))            # waits for the coverage kernels, which read the table it replaces
        assert ev.query()
        second = check(c, bases, offsets, 1, 4, what="after an add")   # the directory was rebuilt
        assert not np.array_equal(first[0], second[0].astype(np.uint32))
        c.coverage_tensors(tb, to, 1, 4)
        c.add_tensors(tb, to)              # ordered on the stream after them
        check(c, bases, offsets, 1, 4, what="after a device add")
        # a failed add (a scratch that cannot be allocated) leaves the rows as they were
        before = c.coverage((bases, offsets), 3, 6, True, np.float64)
        L = _lib.load()
        rc = L.ktb_counter_add_device(c._h, tb.data_ptr(), to.data_ptr(), len(offsets) - 1, 0x7FFFFFFF * CT_T, None)
        assert rc == _lib.KTB_ERR_NOMEM
        after = c.coverage((bases, offsets), 3, 6, True, np.float64)
        assert np.array_equal(before[0], after[0]) and np.array_equal(before[1], after[1])
        check(c, bases, offsets, 3, 6, what="after a failed add")


# ----------------------------------------------------------------------------------------------------------- CLI
def cov(*args, **kw):
    return subprocess.run([str(BIN), "cov", *map(str, args)], capture_output=True, **kw)


def cli_want(path, counted, k, w=16, c=16):
    bases, offsets = read_fastx(path)
    cb, co = read_fastx(counted)
    with KmerCounter(k) as ctr:
        ctr.add((cb, co))
        keys, counts = ctr.result()
    rows, totals = coverage_rows(bases, offsets, keys, counts, k, True, w, c)
    return oracle.format_rows(expected(rows, totals, True, np.float64), norm=True)


@pytest.mark.parametrize("fname", ["reads.fa", "reads.fq", "reads.fq.gz"])
@pytest.mark.parametrize("k", [10, 31])
def test_cli_golden(golden, tmp_path, fname, k):
    out = tmp_path / "cov.txt"
    r = cov("-i", golden / fname, "-o", out, "-k", k)
    assert r.returncode == 0 and r.stderr == b"", r.stderr
    assert out.read_bytes() == cli_want(golden / fname, golden / fname, k)
    other = golden / ("reads.fq" if fname == "reads.fa" else "reads.fa")
    for t in (1, 8):
        r = cov("-i", golden / fname, "-o", out, "-k", k, "-a", other, "-w", 1, "-c", 5, "-t", t, "-m", 2)
        assert r.returncode == 0 and r.stderr == b"", r.stderr
        assert out.read_bytes() == cli_want(golden / fname, other, k, 1, 5)


def test_cli_many_batches_and_stdin(tmp_path):
    rng = np.random.default_rng(12)
    lens = [150] * 120_000 + [30_000_000] + [150] * 30_000   # three 32 MB batches: the long record is one of its own
    bases, offsets = random_batch(rng, lens, n_runs=0.1)
    fq = tmp_path / "big.fq"
    with open(fq, "wb") as f:
        for i in range(len(lens)):
            s = bases[int(offsets[i]):int(offsets[i + 1])].tobytes()
            f.write(b"@r%d\n%s\n+\n%s\n" % (i, s, b"I" * len(s)))
    small = tmp_path / "small.fa"
    small.write_bytes(b"".join(b">s%d\n%s\n" % (i, bases[i * 150:i * 150 + 150].tobytes()) for i in range(3000)))
    out = tmp_path / "cov.txt"
    r = cov("-i", fq, "-o", out, "-k", 21, "-w", 1, "-c", 4)
    assert r.returncode == 0 and r.stderr == b"", r.stderr
    with KmerCounter(21) as ctr:
        ctr.add((bases, offsets))
        keys, counts = ctr.result()
    rows, totals = coverage_rows(bases, offsets, keys, counts, 21, True, 1, 4)
    assert out.read_bytes() == oracle.format_rows(expected(rows, totals, True, np.float64), norm=True)
    # the table from a pipe (-a -), the rows of a file
    with open(fq, "rb") as f:
        r = cov("-i", small, "-o", out, "-k", 21, "-a", "-", "-w", 1, "-c", 4, stdin=f)
    assert r.returncode == 0 and r.stderr == b"", r.stderr
    sb, so = read_fastx(small)
    rows, totals = coverage_rows(sb, so, keys, counts, 21, True, 1, 4)
    assert out.read_bytes() == oracle.format_rows(expected(rows, totals, True, np.float64), norm=True)
    r = cov("-i", tmp_path / "nope.fq", "-o", out, "-k", 21)
    assert r.returncode == 0 and r.stderr.startswith(b"Error:")

