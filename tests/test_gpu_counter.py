"""Batch-wide k-mer counting on the GPU (ktb_counter_*, KmerCounter, `kmertools ctr`): parity with the oracle's windows
counted with np.unique, cross-checks with the sparse and dense rows at scale, skewed input, split and order
independence, u64 counts, the host chunking, the device entry point, the reads and the CLI."""
import ctypes as C
import subprocess
import threading
from pathlib import Path

import numpy as np
import pytest

from kmertools_b200 import KmerCounter, _lib
from kmertools_b200.io import read_fastx

from tests.test_counter_host import count_table, pack
from tests.util import random_batch

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

ROOT = Path(__file__).resolve().parent.parent
BIN = ROOT / "kmertools_b200" / "bin" / "kmertools"
DEV = torch.device("cuda", 0)
PARITY_K = [1, 2, 3, 4, 5, 8, 11, 12, 13, 16, 17, 21, 28, 29, 31]


def on_device(bases, offsets):
    return torch.from_numpy(np.ascontiguousarray(bases)).to(DEV), torch.from_numpy(offsets.astype(np.int64)).to(DEV)


def assert_table(counter, want):
    keys, counts = counter.result()
    assert np.array_equal(keys, want[0]), "keys differ"
    assert np.array_equal(counts, want[1]), "counts differ"
    assert counter.windows == want[2] == int(counts.sum())
    assert len(counter) == len(want[0])


def sum_by_code(codes, values):
    """Distinct codes (ascending) and the sum of their values, on the GPU."""
    u, inv = torch.unique(codes, return_inverse=True)
    s = torch.zeros(len(u), dtype=torch.int64, device=codes.device)
    s.index_add_(0, inv, values.to(torch.int64))
    return u, s


@pytest.mark.parametrize("k", PARITY_K)
@pytest.mark.parametrize("canonical", [True, False])
def test_parity_with_the_oracle(k, canonical):
    rng = np.random.default_rng(100 * k + int(canonical))
    lens = [0, 1, k - 1, k, k + 1, 0, 4095, 4096, 4097, 3 * 4096 + 17] + list(rng.integers(0, 400, size=40))
    bases, offsets = random_batch(rng, lens, noise=0.03, n_runs=0.3)
    want = count_table(bases, offsets, k, canonical)
    with KmerCounter(k, canonical) as c:
        c.add((bases, offsets))
        assert_table(c, want)
    with KmerCounter(k, canonical) as c:
        c.add_tensors(*on_device(bases, offsets))
        assert_table(c, want)


@pytest.fixture(scope="module")
def reads_1m():
    import bench
    return bench.make_workload_torch(bench.WORKLOADS["reads150_k5"], 0.1, DEV)


def sparse_codes_values(tb, to, k, mins):
    """Codes and u32 counts of the sparse rows of a batch, from ktb_sparse_vectorise_device itself: a
    torch.sparse_csr_tensor of 4^31 columns has more elements than int64 can count."""
    n, total = to.numel() - 1, tb.numel()
    row_ptr = torch.empty(n + 1, dtype=torch.int64, device=DEV)
    codes = torch.empty(total, dtype=torch.int64, device=DEV)
    values = torch.empty(total, dtype=torch.int32, device=DEV)
    stream = torch.cuda.current_stream(DEV).cuda_stream
    _lib.check(_lib.load().ktb_sparse_vectorise_device(
        tb.data_ptr(), to.data_ptr(), n, total, k, int(mins), _lib.NORM_COUNTS, _lib.OUT_U32, row_ptr.data_ptr(),
        codes.data_ptr(), values.data_ptr(), total, None, stream))
    nnz = int(row_ptr[-1])
    return codes[:nnz], values[:nnz]


@pytest.mark.parametrize("k", [21, 31])
def test_equals_the_sparse_rows_summed_at_scale(reads_1m, k):
    tb, to = reads_1m
    assert to.numel() - 1 == 1_000_000
    for mins in (True, False):
        u, s = sum_by_code(*sparse_codes_values(tb, to, k, mins))
        with KmerCounter(k, mins) as c:
            c.add_tensors(tb, to)
            keys, counts = c.result_tensors()
            assert torch.equal(keys, u) and torch.equal(counts, s)
            assert c.windows == int(s.sum())
        del u, s


@pytest.mark.parametrize("k,nreads", [(5, 1_000_000), (8, 20_000), (12, 100)])
def test_equals_the_dense_column_sums(reads_1m, k, nreads):
    from kmertools_b200 import OligoComputer
    tb, to = reads_1m
    sub_o = to[:nreads + 1].contiguous()
    sub_b = tb[:int(sub_o[-1])].contiguous()
    oc = OligoComputer(k)
    _, p2k, _ = oc.kmer_pos_maps()
    for mins in (True, False):
        rows = oc.vectorise_tensors(sub_b, sub_o, norm_mode=0, mins=mins, dtype=torch.int32)
        sums = rows.to(torch.int64).sum(0)
        del rows
        codes = torch.from_numpy(p2k.astype(np.int64)).to(DEV) if mins else torch.arange(4 ** k, device=DEV)
        nz = sums > 0
        order = torch.argsort(codes[nz])
        with KmerCounter(k, mins) as c:
            c.add_tensors(sub_b, sub_o)
            keys, counts = c.result_tensors()
        assert torch.equal(keys, codes[nz][order]) and torch.equal(counts, sums[nz][order])
    oc.close()


def test_skewed_input():
    n = 10 ** 8
    with KmerCounter(21) as c:   # one key: AAA... and its reverse complement TTT... share code 0
        c.add((np.full(n, ord("A"), np.uint8), np.array([0, n], np.uint64)))
        keys, counts = c.result()
        assert keys.tolist() == [0] and counts.tolist() == [n - 20] and c.windows == n - 20
    rng = np.random.default_rng(7)
    for unit in (b"AC", b"ACGTTGA"):
        seq = unit * (1_000_000 // len(unit))
        bases, offsets = pack([seq, seq[3:500_000]])
        for k in (1, 4, 13, 31):
            for mins in (True, False):
                with KmerCounter(k, mins) as c:
                    c.add((bases, offsets))
                    assert_table(c, count_table(bases, offsets, k, mins))
    amb = np.frombuffer(b"NRYKMSWBDHVn-." * 100_000, np.uint8)
    with KmerCounter(5) as c:
        c.add((amb, np.array([0, len(amb) // 2, len(amb)], np.uint64)))
        assert len(c) == 0 and c.windows == 0
        keys, counts = c.result()
        assert keys.size == 0 and counts.size == 0
    bases, offsets = random_batch(rng, [2_000_000])
    with KmerCounter(31) as c:   # nearly every key distinct
        c.add_tensors(*on_device(bases, offsets))
        want = count_table(bases, offsets, 31)
        assert len(want[0]) > 1_990_000
        assert_table(c, want)


def test_split_and_order_independence():
    rng = np.random.default_rng(11)
    lens = list(rng.integers(0, 3000, size=600)) + [0, 5, 20_000]
    bases, offsets = random_batch(rng, lens, noise=0.02, n_runs=0.2)
    n = len(lens)
    for k in (3, 21):
        want = count_table(bases, offsets, k)
        tables = []
        for parts in (1, 2, 7):
            cuts = np.sort(rng.choice(np.arange(1, n), size=parts - 1, replace=False)) if parts > 1 else []
            bounds = [0, *cuts, n]
            pieces = [(bounds[i], bounds[i + 1]) for i in range(parts)]
            rng.shuffle(pieces)
            with KmerCounter(k) as c:
                c.add([])                                                      # n = 0
                c.add_tensors(torch.zeros(0, dtype=torch.uint8, device=DEV), torch.zeros(1, dtype=torch.int64, device=DEV))
                c.add(["", "AC"])                                              # nothing valid at k >= 3
                assert len(c) == 0 and c.windows == 0
                for i, (a, b) in enumerate(pieces):
                    o = offsets[a:b + 1] - offsets[a]
                    bb = bases[int(offsets[a]):int(offsets[b])]
                    if i % 2:
                        c.add_tensors(*on_device(bb, o))
                    else:
                        c.add((bb, o))
                tables.append(c.result())
                assert c.windows == want[2]
        for t in tables:
            assert np.array_equal(t[0], want[0]) and np.array_equal(t[1], want[1])


@pytest.mark.parametrize("k", [1, 31])
def test_counts_past_2_pow_32(k):
    n = 1 << 30
    tb = torch.full((n,), ord("A"), dtype=torch.uint8, device=DEV)
    to = torch.tensor([0, n], dtype=torch.int64, device=DEV)
    with KmerCounter(k) as c:
        for _ in range(5):
            c.add_tensors(tb, to)
        keys, counts = c.result()
        want = 5 * (n - k + 1)
        assert want > 2 ** 32
        assert keys.tolist() == [0] and counts.tolist() == [want] and c.windows == want
    del tb
    torch.cuda.empty_cache()


def test_host_chunks_equal_the_device_entry():
    """Several 2^26-base chunks, one sequence longer than a chunk in the middle."""
    rng = np.random.default_rng(5)
    lens = [150] * 300_000 + [70_000_000] + list(rng.integers(0, 1000, size=200_000)) + [7]
    bases, offsets = random_batch(rng, lens, noise=0.001, n_runs=0.01)
    assert offsets[-1] > 3 * (1 << 26)
    for k in (2, 21):
        with KmerCounter(k) as h, KmerCounter(k) as d:
            h.add((bases, offsets))
            d.add_tensors(*on_device(bases, offsets))
            a, b = h.result(), d.result()
            assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) and h.windows == d.windows


def test_device_entry_point():
    rng = np.random.default_rng(9)
    bases, offsets = random_batch(rng, list(rng.integers(0, 600, size=500)) + [0, 9000], noise=0.02)
    want = count_table(bases, offsets, 17)
    # a batch inside a larger buffer: offsets[0] > 0 and bytes on both sides that must not be read
    pad = np.frombuffer(b"ACGT" * 2500, np.uint8)
    buf = np.concatenate([pad, bases, pad])
    tb, to = on_device(buf, offsets + len(pad))
    L = _lib.load()
    s = torch.cuda.Stream(DEV)
    with KmerCounter(17) as c:
        with torch.cuda.stream(s):
            _lib.check(L.ktb_counter_add_device(c._h, tb.data_ptr(), to.data_ptr(), len(offsets) - 1,
                                                int(to[-1]), s.cuda_stream))
        assert_table(c, want)
    # back to back on a non-default stream, no host synchronisation between the adds
    tb2, to2 = on_device(bases, offsets)
    with KmerCounter(17) as c, torch.cuda.stream(s):
        for _ in range(3):
            c.add_tensors(tb2, to2)
        keys, counts = c.result_tensors()
        s.synchronize()
        assert np.array_equal(keys.cpu().numpy().astype(np.uint64), want[0])
        assert np.array_equal(counts.cpu().numpy().astype(np.uint64), 3 * want[1])
    # two counters on two streams at once
    other = random_batch(rng, list(rng.integers(0, 5000, size=400)))
    wants = [want, count_table(*other, 17)]
    batches = [(tb2, to2), on_device(*other)]
    counters = [KmerCounter(17), KmerCounter(17)]
    streams = [torch.cuda.Stream(DEV), torch.cuda.Stream(DEV)]

    def work(i):
        with torch.cuda.stream(streams[i]):
            for _ in range(4):
                counters[i].add_tensors(*batches[i])

    threads = [threading.Thread(target=work, args=(i,)) for i in range(2)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    for c, w in zip(counters, wants):
        keys, counts = c.result()
        assert np.array_equal(keys, w[0]) and np.array_equal(counts, 4 * w[1])
        c.close()


def test_reads_respect_cap():
    rng = np.random.default_rng(3)
    bases, offsets = random_batch(rng, list(rng.integers(0, 300, size=200)))
    L = _lib.load()
    with KmerCounter(9) as c:
        c.add((bases, offsets))
        keys, counts = c.result()
        nk = len(keys)
        assert nk > 10
        tk, tc = c.result_tensors()
        assert np.array_equal(tk.cpu().numpy().astype(np.uint64), keys)
        assert np.array_equal(tc.cpu().numpy().astype(np.uint64), counts)
        sentinel = 0xDEADBEEFCAFEF00D
        for cap in (0, 1, nk - 1, nk, nk + 1):
            m = min(cap, nk)
            hk = np.full(nk + 4, sentinel, np.uint64)
            hc = np.full(nk + 4, sentinel, np.uint64)
            _lib.check(L.ktb_counter_read(c._h, hk.ctypes.data, hc.ctypes.data, cap))
            assert np.array_equal(hk[:m], keys[:m]) and np.array_equal(hc[:m], counts[:m])
            assert np.all(hk[m:] == sentinel) and np.all(hc[m:] == sentinel)
            dk = torch.full((nk + 4,), -7, dtype=torch.int64, device=DEV)
            dc = torch.full((nk + 4,), -7, dtype=torch.int64, device=DEV)
            _lib.check(L.ktb_counter_read_device(c._h, dk.data_ptr(), dc.data_ptr(), cap, None))
            torch.cuda.synchronize()
            assert np.array_equal(dk[:m].cpu().numpy().astype(np.uint64), keys[:m])
            assert np.array_equal(dc[:m].cpu().numpy().astype(np.uint64), counts[:m])
            assert bool((dk[m:] == -7).all()) and bool((dc[m:] == -7).all())
        _lib.check(L.ktb_counter_read(c._h, None, None, 0))
        _lib.check(L.ktb_counter_read_device(c._h, None, None, 0, None))


def ctr(*args):
    return subprocess.run([str(BIN), "ctr", *map(str, args)], capture_output=True, text=True)


def read_lines(path):
    text = Path(path).read_text()
    assert text == "" or text.endswith("\n")
    return [ln.split("\t") for ln in text.splitlines()]


@pytest.mark.parametrize("fname", ["reads.fa", "reads.fq", "reads.fq.gz"])
@pytest.mark.parametrize("k", [10, 15, 31])
def test_cli_golden(golden, tmp_path, fname, k):
    from pykmertools.utils import to_acgt
    bases, offsets = read_fastx(golden / fname)
    keys, counts, _ = count_table(bases, offsets, k)
    out = tmp_path / "out"
    r = ctr("-i", golden / fname, "-o", out, "-k", k)
    assert r.returncode == 0 and r.stderr == "", r.stderr
    lines = read_lines(out / "kmers.counts")
    assert [int(a) for a, _ in lines] == keys.tolist() and [int(b) for _, b in lines] == counts.tolist()
    r = ctr("-i", golden / fname, "-o", out, "-k", k, "--acgt", "-t", 3, "-m", 4)
    assert r.returncode == 0 and r.stderr == "", r.stderr
    lines = read_lines(out / "kmers.counts")
    assert [a for a, _ in lines] == [to_acgt(int(x), k) for x in keys]
    assert [int(b) for _, b in lines] == counts.tolist()


def test_cli_many_batches(tmp_path):
    """Several driver batches (32 MB of bases each) and one record larger than a batch, against KmerCounter."""
    rng = np.random.default_rng(21)
    lens = [150] * 250_000 + [40_000_000] + [150] * 100_000
    bases, offsets = random_batch(rng, lens, n_runs=0.1)
    fq = tmp_path / "big.fq"
    with open(fq, "wb") as f:
        for i in range(len(lens)):
            s = bases[int(offsets[i]):int(offsets[i + 1])].tobytes()
            f.write(b"@r%d\n%s\n+\n%s\n" % (i, s, b"I" * len(s)))
    r = ctr("-i", fq, "-o", tmp_path / "o", "-k", 25)
    assert r.returncode == 0 and r.stderr == "", r.stderr
    with KmerCounter(25) as c:
        c.add((bases, offsets))
        keys, counts = c.result()
    text = (tmp_path / "o" / "kmers.counts").read_bytes()
    want = "".join(f"{a}\t{b}\n" for a, b in zip(keys.tolist(), counts.tolist())).encode()
    assert text == want
    r = ctr("-i", tmp_path / "nope.fq", "-o", tmp_path / "o2", "-k", 25)
    assert r.returncode == 0 and r.stderr.startswith("Error:")
