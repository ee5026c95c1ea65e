"""The file drivers (`ktb_comp_oligo_file`, `ktb_comp_cgr_file`, `kmertools comp oligo|cgr`) compared byte for byte, whole
file, with text built independently of them: rounding ties through the GPU text formatter (`format_norm_kernel`), every
k the library accepts across at least three batches, many batches through every writer and formatter thread count,
cached buffer sets and concurrent callers, and k-mer CGR with a bound on the formatter's memory.

Batch geometry (file_api.cu): a batch holds at most 64 MiB of output rows (9 bytes a value for normalised text, 4 for
counts, 8 for normalised CGR), at most 4 Mi records and 32 MiB of bases."""
import os
import subprocess
import threading
from decimal import ROUND_HALF_EVEN, Decimal
from pathlib import Path

import numpy as np
import pytest

from oracle import oracle as O
from tests.util import ALPHA

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parent.parent
BIN = ROOT / "kmertools_b200" / "bin" / "kmertools"
OUT_CAP = 64 << 20


def kio():
    from kmertools_b200 import io
    return io


def cli(sub, args, env=None, **kw):
    e = dict(os.environ)
    e.pop("KTB_WRITER", None)
    e.update(env or {})
    return subprocess.run([str(BIN), "comp", sub, *map(str, args)], capture_output=True, env=e, **kw)


def rows_per_batch(k, canonical, norm, cgr=False):
    d = O.dim(k, canonical or cgr)
    per = d * (8 if cgr else 9) if norm else d * 4
    return max(1, min(OUT_CAP // per, 4 << 20))


def write_fastx(path, bases, offsets, fastq=False):
    """Records "r" of bases[offsets[i]:offsets[i+1]], one line each (FASTQ with quality 'I').  A FASTQ record with an
    empty sequence has an empty quality string, which the reader rejects (test_io_host.py::
    test_fastq_errors_follow_the_reader), so FASTQ records here are never empty."""
    lens = np.diff(offsets.astype(np.int64))
    assert not fastq or lens.min(initial=1) > 0
    head = b"@r\n" if fastq else b">r\n"
    rec = len(head) + lens + 1 + ((lens + 3) if fastq else 0)
    starts = np.zeros(len(lens) + 1, dtype=np.int64)
    np.cumsum(rec, out=starts[1:])
    out = np.empty(int(starts[-1]), dtype=np.uint8)
    s = starts[:-1]
    for i, ch in enumerate(head):
        out[s + i] = ch
    total = int(offsets[-1] - offsets[0])
    dest = np.arange(total, dtype=np.int64) + np.repeat(s + len(head) - (offsets[:-1].astype(np.int64) - int(offsets[0])), lens)
    out[dest] = bases[int(offsets[0]):int(offsets[-1])]
    nl = s + len(head) + lens
    out[nl] = ord("\n")
    if fastq:
        out[nl + 1] = ord("+")
        out[nl + 2] = ord("\n")
        out[dest + lens.repeat(lens) + 3] = ord("I")
        out[starts[1:] - 1] = ord("\n")
    out.tofile(path)


def mixed_batch(rng, lengths, n_runs=0.05):
    """ACGT with lower case, IUPAC bytes and N runs (nothing that ends a FASTA line)."""
    lengths = np.asarray(lengths, dtype=np.int64)
    offsets = np.zeros(len(lengths) + 1, dtype=np.uint64)
    np.cumsum(lengths, out=offsets[1:])
    bases = ALPHA[rng.integers(0, 4, size=int(offsets[-1]))]
    m = rng.random(bases.size)
    bases[m < 0.01] += 32                                          # acgt
    bases[m > 0.998] = np.frombuffer(b"NRYKMn", dtype=np.uint8)[rng.integers(0, 6, size=int((m > 0.998).sum()))]
    for i in np.nonzero(rng.random(len(lengths)) < n_runs)[0]:
        L = int(lengths[i])
        if L:
            a = int(rng.integers(0, L))
            bases[int(offsets[i]) + a:int(offsets[i]) + min(L, a + int(rng.integers(1, max(2, L // 3))))] = ord("N")
    return bases, offsets


def header_line(k, canonical, delim):
    return (delim.join(O.header(k, canonical)) + "\n").encode()


def assert_same_file(got, want, head=b""):
    """got == head + want, compared in chunks; `want` is a path or bytes.  The first difference is reported."""
    got = Path(got)
    want_size = Path(want).stat().st_size if isinstance(want, Path) else len(want)
    assert got.stat().st_size == len(head) + want_size, (got.stat().st_size, len(head) + want_size)
    step = 32 << 20
    with open(got, "rb") as g:
        assert g.read(len(head)) == head, "header line"
        wf = open(want, "rb") if isinstance(want, Path) else None
        try:
            pos = 0
            while pos < want_size:
                a = g.read(step)
                b = wf.read(step) if wf else want[pos:pos + step]
                if a != b:
                    i = next(j for j in range(len(a)) if a[j] != b[j])
                    raise AssertionError(f"first difference at byte {pos + i} of the body: got {a[max(0, i - 40):i + 40]!r}, "
                                         f"want {b[max(0, i - 40):i + 40]!r}")
                pos += len(a)
        finally:
            if wf:
                wf.close()


def oracle_text(path, bases, offsets, k, canonical=True, norm=True, delim=" "):
    """The oracle's text of the records (composition/src/oligo.rs:126-144), written to `path`."""
    O.baseline_text(bases, offsets, k, canonical, norm, delim, path=str(path))
    return Path(path)


# ----------------------------------------------------------------------------- a. ties and near-ties

def _q6(c, d):
    """Rust's {:.6} of the f64 quotient c / d: Python's `/` is the same correctly rounded IEEE division, and Decimal
    holds the exact binary value of the double it is given."""
    return str(Decimal(c / d).quantize(Decimal("0.000001"), rounding=ROUND_HALF_EVEN)) if d else "0.000000"


def _tie_cases():
    """(c, d) pairs: a record of c A's then d - c C's has k = 1 rows (c/d, (d-c)/d) canonical, (c/d, (d-c)/d, 0, 0) raw."""
    rng = np.random.default_rng(128)
    cases = []
    # exact decimal ties: c odd, d = 2^7 * 5^b makes c/d * 10^6 = c * 5^(6-b) / 2.  Where 5 divides d the quotient is
    # not exact in binary, so the digit follows the last bit of the division.
    for b, d in enumerate((128, 640, 3200, 16000, 80000, 400000, 2000000)):
        odd = np.arange(1, d, 2)
        cs = odd if d <= 3200 else np.r_[odd[:2], odd[-2:], rng.choice(odd[2:-2], size=(96, 40, 16, 4)[b - 3], replace=False)]
        cases += [(int(c), d) for c in cs]
    # near-ties: the c whose c * 10^6 mod d is closest to d / 2 without being equal (and its neighbours where short)
    for d in (3, 7, 11, 97, 1001, 4099, 65537, 999983, (1 << 23) - 1, (1 << 23) + 1, (1 << 24) - 1, (1 << 24) + 1,
              (1 << 24) + 3):
        c = np.arange(1, d, dtype=np.int64)
        dist = np.abs(2 * ((c * 1_000_000) % d) - d)
        dist[dist == 0] = d + 1
        best = int(c[np.argmin(dist)])
        cases += [(x, d) for x in ((best - 1, best, best + 1) if d < 1 << 20 else (best,)) if 0 < x < d]
    cases += [(1, 1), (5, 5), (0, 9), (0, 0)]
    return cases


def test_rounding_ties_through_the_gpu_formatter(tmp_path):
    cases = _tie_cases()
    fa = tmp_path / "ties.fa"
    with open(fa, "wb") as fh:
        for c, d in cases:
            fh.write(b">r\n" + b"A" * c + b"C" * (d - c) + b"\n")
        fh.write(b">allN\n" + b"N" * 1000 + b"\n")
    want_canon = "".join(f"{_q6(c, d)} {_q6(d - c, d)}\n" for c, d in cases) + "0.000000 0.000000\n"
    want_raw = "".join(f"{_q6(c, d)} {_q6(d - c, d)} 0.000000 0.000000\n" for c, d in cases) + \
        "0.000000 0.000000 0.000000 0.000000\n"
    assert "0.007812 0.992188\n" in want_canon and "0.023438 0.976562\n" in want_canon   # 1/128 down, 3/128 up
    out = tmp_path / "o"
    for canonical, want in ((True, want_canon.encode()), (False, want_raw.encode())):
        assert want == O.comp_oligo_text(fa, 1, canonical=canonical)
        kio().comp_oligo(fa, out, k=1, raw_count=not canonical)
        assert_same_file(out, want)
        r = cli("oligo", ["-i", fa, "-o", out, "--any-k", "-k", 1] + ([] if canonical else ["-r"]))
        assert r.returncode == 0 and r.stderr == b"", r.stderr
        assert_same_file(out, want)
    out.unlink()


# ----------------------------------------------------------------------------- b. every k, across batches

MODES = (  # canonical, norm, delim, header
    (True, True, " ", False), (True, False, ",", True), (False, True, ",", True), (False, False, " ", False))
MAX_LEN = {1: 8, 2: 12, 8: 400, 9: 400, 10: 400, 11: 3000, 12: 3000}
LONG = {1: 2000, 2: 4000, 8: 20_000, 9: 30_000, 10: 40_000, 11: 20_000, 12: 20_000}


def _every_k_modes(k):
    """(canonical, norm, delim, header, records): enough records for three batches; -H and csv at k = 1, 2 and 8."""
    out = []
    for canonical, norm, delim, header in MODES:
        if not canonical and k > 10:
            continue
        if k not in (1, 2, 8):
            delim, header = " ", False
        r = rows_per_batch(k, canonical, norm)
        out.append((canonical, norm, delim, header, 2 * r + min(r, 7)))
    return out


@pytest.mark.parametrize("k", [1, 2, 8, 9, 10, 11, 12])
def test_every_k_across_batches(tmp_path, k):
    """Each mode's file is a prefix of one record set, three batches long.  The last record of every prefix is its
    longest, so the driver's per-handle scratch (the bucket pool at k >= 9 canonical and k >= 8 raw) grows in a
    later batch; records are mixed lengths with N runs, lower case and IUPAC bytes."""
    modes = _every_k_modes(k)
    n = max(m[4] for m in modes)
    rng = np.random.default_rng(1000 + k)
    lengths = rng.integers(0, MAX_LEN[k], size=n)
    lengths[rng.random(n) < 0.02] = 0
    for j, m in enumerate(sorted(m[4] for m in modes)):
        lengths[m - 1] = LONG[k] * (j + 1)
    bases, offsets = mixed_batch(rng, lengths, n_runs=0.05 if n < 100_000 else 0.002)
    out, want = tmp_path / "o", tmp_path / "want"
    for canonical, norm, delim, header, m in modes:
        fa = tmp_path / "in.fa"
        write_fastx(fa, bases, offsets[:m + 1])
        sub = (bases, offsets[:m + 1])
        oracle_text(want, *sub, k, canonical, norm, delim)
        head = header_line(k, canonical, delim) if header else b""
        st = kio().comp_oligo(fa, out, k=k, counts=not norm, raw_count=not canonical,
                              preset={" ": "spc", ",": "csv"}[delim], header=header)
        assert st["records"] == m
        assert_same_file(out, want, head)
        if k == 9 and canonical and norm:
            r = cli("oligo", ["-i", fa, "-o", out, "--any-k", "-k", k, "-t", 3])
            assert r.returncode == 0 and r.stderr == b"", r.stderr
            assert_same_file(out, want)
        out.unlink()
    want.unlink()


def test_k13_is_refused(golden, tmp_path):
    out = tmp_path / "o"
    r = cli("oligo", ["-i", golden / "reads.fa", "-o", out, "--any-k", "-k", 13])
    assert r.returncode == 0 and r.stderr.startswith(b"Error: "), r.stderr   # printed, exit 0, like args.rs:260-262
    assert not out.exists()
    assert cli("oligo", ["-i", golden / "reads.fa", "-o", out, "-k", 13]).returncode == 2


# ----------------------------------------------------------------------------- c. many batches, threads, writers

@pytest.fixture(scope="module")
def reads3000(tmp_path_factory):
    """~3,000 reads at k = 7: 4 normalised text batches (910 rows each), 2 counts batches (2,048 rows each)."""
    d = tmp_path_factory.mktemp("reads3000")
    rng = np.random.default_rng(3000)
    lengths = np.r_[rng.integers(1, 400, size=2000), [60_000], rng.integers(1, 400, size=1000)]
    bases, offsets = mixed_batch(rng, lengths)
    fq = d / "reads.fq"
    write_fastx(fq, bases, offsets, fastq=True)
    assert len(lengths) > 3 * rows_per_batch(7, True, True) and len(lengths) > rows_per_batch(7, True, False)
    return fq, oracle_text(d / "norm", bases, offsets, 7), oracle_text(d / "counts", bases, offsets, 7, norm=False)


@pytest.mark.parametrize("norm", [True, False], ids=["norm", "counts"])
def test_threads_and_writers_across_batches(reads3000, tmp_path, norm):
    fq, want_norm, want_counts = reads3000
    want = want_norm if norm else want_counts
    out = tmp_path / "o"
    for threads in (1, 3, 8):
        for writer in ("map", "seq"):
            r = cli("oligo", ["-i", fq, "-o", out, "-k", 7, "-t", threads] + ([] if norm else ["-c"]),
                    env={"KTB_WRITER": writer})
            assert r.returncode == 0 and r.stderr == b"", (threads, writer, r.stderr)
            assert_same_file(out, want)
            out.unlink()


def test_stdout_pipe_falls_back_to_sequential_writes(reads3000):
    fq, want, _ = reads3000
    r = cli("oligo", ["-i", fq, "-o", "/dev/stdout", "-k", 7], env={"KTB_WRITER": "map"})
    assert r.returncode == 0 and r.stderr == b"", r.stderr
    assert r.stdout == want.read_bytes()


def test_empty_inputs(tmp_path):
    out = tmp_path / "o"
    empty = tmp_path / "empty.fa"
    empty.write_bytes(b"")
    for flags, want in (([], b""), (["-H"], header_line(4, True, " ")), (["-c", "-H", "-p", "csv"], header_line(4, True, ","))):
        r = cli("oligo", ["-i", empty, "-o", out, "-k", 4, *flags])
        assert r.returncode == 0 and r.stderr == b"", r.stderr
        assert out.read_bytes() == want, flags
    r = cli("oligo", ["-i", "-", "-o", out, "-k", 4], input=b"")
    assert r.returncode == 0 and r.stderr == b"" and out.read_bytes() == b""
    blank = tmp_path / "blank.fa"
    blank.write_bytes(b">a\n>b\n\n>c\n")
    for flags, kw in (([], {}), (["-c", "-r"], {"norm": False, "canonical": False})):
        r = cli("oligo", ["-i", blank, "-o", out, "-k", 4, *flags])
        assert r.returncode == 0 and r.stderr == b"", r.stderr
        want = O.comp_oligo_text(blank, 4, **kw)
        assert want.count(b"\n") == 3 and out.read_bytes() == want, flags
    r = cli("cgr", ["-i", blank, "-o", out, "-k", 3])
    assert r.returncode == 0 and out.read_bytes() == O.comp_cgr_text(blank, 3, 9)


# ----------------------------------------------------------------------------- d. cached buffer sets, concurrent callers

def _small_fasta(path, seed, lengths):
    bases, offsets = mixed_batch(np.random.default_rng(seed), lengths)
    write_fastx(path, bases, offsets)
    return path, bases, offsets


def test_cached_buffer_sets_and_concurrent_callers(tmp_path):
    io = kio()
    out = tmp_path / "o"
    f12, *batch12 = _small_fasta(tmp_path / "k12.fa", 12, [500, 30_000, 1500])
    f3, _, _ = _small_fasta(tmp_path / "k3.fa", 3, np.arange(500) % 300)
    f5, _, _ = _small_fasta(tmp_path / "k5.fa", 5, np.r_[np.arange(300), [200_000]])
    f7, _, _ = _small_fasta(tmp_path / "k7.fa", 7, np.arange(200) * 5)
    io.comp_oligo(f12, out, k=12)                      # the largest buffers go to the cache ...
    assert_same_file(out, oracle_text(tmp_path / "want12", *batch12, 12))
    io.comp_oligo(f3, out, k=3, counts=True)            # ... and are reused by smaller runs of another kind
    assert_same_file(out, O.comp_oligo_text(f3, 3, norm=False))
    io.comp_cgr(f5, out, k=5)
    assert_same_file(out, O.comp_cgr_text(f5, 5, 25))
    io.release_cached_buffers()
    io.comp_oligo(f7, out, k=7)
    assert_same_file(out, O.comp_oligo_text(f7, 7))

    out_a, out_b, errors = tmp_path / "a", tmp_path / "b", []

    def call(fn):
        try:
            fn()
        except Exception as exc:   # noqa: BLE001 - re-raised on the main thread
            errors.append(exc)

    want_a, want_b = O.comp_oligo_text(f7, 6, canonical=False), O.comp_cgr_text(f5, 4, 16, norm=False)
    for _ in range(3):
        th = [threading.Thread(target=call, args=(lambda: io.comp_oligo(f7, out_a, k=6, raw_count=True),)),
              threading.Thread(target=call, args=(lambda: io.comp_cgr(f5, out_b, k=4, counts=True, threads=3),))]
        for t in th:
            t.start()
        for t in th:
            t.join()
        assert not errors, errors
        assert_same_file(out_a, want_a)
        assert_same_file(out_b, want_b)


# ----------------------------------------------------------------------------- e. k-mer CGR

@pytest.fixture(scope="module")
def cgr_small(tmp_path_factory):
    """Short and medium records, an N run, and long near-homopolymers whose rare k-mers have frequencies below 1e-5."""
    d = tmp_path_factory.mktemp("cgr")
    rng = np.random.default_rng(55)
    recs = [b"", b"AC", b"ACGTNNNNACGT", b"N" * 50]
    recs += [ALPHA[rng.integers(0, 4, size=n)].tobytes() for n in (7, 8, 9, 150, 1000, 70_000)]
    recs += [b"A" * 150_000 + b"CG" + b"A" * 100_000, b"ACGT" * 40_000 + b"T" + b"ACGT" * 30_000]
    fa = d / "cgr.fa"
    with open(fa, "wb") as fh:
        for s in recs:
            fh.write(b">r\n" + s + b"\n")
    return fa


def _cgr_check(fa, out, k, vec, norm, via_cli, threads=0):
    want = O.comp_cgr_text(fa, k, k * k if vec is None else vec, norm)
    if via_cli:
        args = ["-i", fa, "-o", out, "-k", k, "-t", threads] + ([] if vec is None else ["-v", vec]) + ([] if norm else ["-c"])
        r = cli("cgr", args)
        assert r.returncode == 0 and r.stderr == b"", r.stderr
    else:
        kio().comp_cgr(fa, out, k=k, counts=not norm, vec_size=vec, threads=threads)
    assert_same_file(out, want)
    return want


@pytest.mark.parametrize("k", [1, 2, 3, 4, 5, 6, 7, 8])
def test_cgr_kmer_mode(cgr_small, tmp_path, k):
    out = tmp_path / "o"
    for vec in (None, 1, 7, 1000):
        for norm in (True, False):
            want = _cgr_check(cgr_small, out, k, vec, norm, via_cli=3 <= k <= 7, threads=(0, 2)[vec == 7])
            if norm and k >= 3:
                assert b",0.00000" in want    # a frequency below 1e-5, in fixed notation
            if norm and k == 4 and vec is None:
                assert b"e-" not in want


@pytest.fixture(scope="module")
def cgr_reads(tmp_path_factory):
    """2,500 reads at k = 7: three normalised CGR batches (1,024 rows each) and two counts batches (2,048 rows)."""
    d = tmp_path_factory.mktemp("cgr_reads")
    rng = np.random.default_rng(2500)
    lengths = np.r_[rng.integers(1, 300, size=1500), [50_000], rng.integers(1, 300, size=999)]
    fq = d / "reads.fq"
    write_fastx(fq, *mixed_batch(rng, lengths), fastq=True)
    assert 2 * rows_per_batch(7, True, True, cgr=True) < len(lengths) and rows_per_batch(7, True, False, cgr=True) < len(lengths)
    return fq


@pytest.mark.parametrize("norm", [True, False], ids=["norm", "counts"])
def test_cgr_across_batches(cgr_reads, tmp_path, norm):
    out = tmp_path / "o"
    want = O.comp_cgr_text(cgr_reads, 7, 49, norm)
    for threads in (1, 5):
        r = cli("cgr", ["-i", cgr_reads, "-o", out, "-k", 7, "-t", threads] + ([] if norm else ["-c"]))
        assert r.returncode == 0 and r.stderr == b"", r.stderr
        assert_same_file(out, want)
        out.unlink()


# Peak resident memory that `comp cgr -k 7` over cgr_reads adds to the same command on one short read (the process's
# CUDA context, handle and pinned buffers are in both).  The formatter reserves room for the longest text a row can
# have but touches only what it writes, about 27 bytes a value here: ~230 MB of text per normalised batch of 1,024 rows
# and ~460 MB per counts batch of 2,048 rows, in each of the two buffer sets.  Zero-filling 420 bytes a value touched
# 3.7 GB per normalised batch and 7.5 GB per counts batch.
CGR_MAXRSS_GROWTH_BOUND = 3 << 29


def _cgr_maxrss(fa, out, norm):
    """ru_maxrss in bytes of `comp cgr -k 7 -t 4` on `fa`, from wait4 on the child."""
    p = subprocess.Popen([str(BIN), "comp", "cgr", "-i", str(fa), "-o", str(out), "-k", "7", "-t", "4"] +
                         ([] if norm else ["-c"]), stderr=subprocess.PIPE)
    _, status, ru = os.wait4(p.pid, 0)
    p.returncode = os.waitstatus_to_exitcode(status)
    err = p.stderr.read()
    p.stderr.close()
    assert p.returncode == 0 and err == b"", err
    return ru.ru_maxrss * 1024


@pytest.mark.parametrize("norm", [True, False], ids=["norm", "counts"])
def test_cgr_formatter_memory_is_bounded(cgr_reads, tmp_path, norm):
    one = tmp_path / "one.fq"
    one.write_bytes(b"@r\nACGTACGTAC\n+\nIIIIIIIIII\n")
    out = tmp_path / "o"
    base = _cgr_maxrss(one, out, norm)
    full = _cgr_maxrss(cgr_reads, out, norm)
    print(f"comp cgr -k 7 {'' if norm else '-c '}ru_maxrss: one read {base / 2**20:.0f} MiB, 2,500 reads {full / 2**20:.0f} MiB")
    assert full - base < CGR_MAXRSS_GROWTH_BOUND, (base, full)
    assert out.stat().st_size > 256 << 20
    out.unlink()
