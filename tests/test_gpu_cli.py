"""`kmertools comp oligo` drop-in (C++ CLI over the C ABI) against the reference's golden files and the
oracle.  Restates composition/src/oligo.rs:311-432 (vec_mmap_test, vec_batch_*_test, *_with_header_test)."""
import subprocess
from pathlib import Path

import numpy as np
import pytest

from oracle import oracle as O

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parent.parent
BIN = ROOT / "kmertools_b200" / "bin" / "kmertools"


def run(args, stdin=None):
    return subprocess.run([str(BIN), "comp", "oligo", *map(str, args)], input=stdin, capture_output=True)


@pytest.mark.parametrize("fname", ["reads.fa", "reads.fq", "reads.fq.gz"])
def test_config1_golden_norm(golden, tmp_path, fname):
    """BASELINE config 1: kmertools comp oligo k=4 canonical normalised on the repo fixture."""
    out = tmp_path / "out.kmers"
    r = run(["-i", golden / fname, "-o", out, "-k", 4])
    assert r.returncode == 0 and r.stderr == b"", r.stderr
    assert out.read_bytes() == (golden / "expected_fa.kmers").read_bytes()


def test_golden_counts_header_and_presets(golden, tmp_path):
    out = tmp_path / "o"
    assert run(["-i", golden / "reads.fa", "-o", out, "-k", 4, "-c"]).returncode == 0
    assert out.read_bytes() == (golden / "expected_fa_batch_unnorm.kmers").read_bytes()
    assert run(["-i", golden / "reads.fa", "-o", out, "-k", 4, "-H"]).returncode == 0
    assert out.read_bytes() == (golden / "expected_fa_header.kmers").read_bytes()
    spc = (golden / "expected_fa.kmers").read_bytes()
    run(["-i", golden / "reads.fa", "-o", out, "-k", 4, "-p", "csv"])
    assert out.read_bytes() == spc.replace(b" ", b",")
    run(["-i", golden / "reads.fa", "-o", out, "-k", 4, "--preset", "tsv", "-t", 8])
    assert out.read_bytes() == spc.replace(b" ", b"\t")


def test_stdin_input(golden, tmp_path):
    out = tmp_path / "o"
    r = run(["-i", "-", "-o", out, "-k", 4], stdin=(golden / "reads.fq").read_bytes())
    assert r.returncode == 0
    assert out.read_bytes() == (golden / "expected_fa.kmers").read_bytes()


def test_cli_errors_follow_the_reference(golden, tmp_path):
    r = run(["-i", tmp_path / "nope.fa", "-o", tmp_path / "o", "-k", 4])
    assert r.returncode == 0 and b"Error: Unable to open" in r.stderr     # args.rs:260-262 prints, exits 0
    assert run(["-i", golden / "reads.fa", "-o", tmp_path / "o", "-k", 9]).returncode == 2   # clap range 3..=7
    assert run(["-i", golden / "reads.fa"]).returncode == 2


@pytest.mark.parametrize("k", [3, 4, 5, 6, 7])
def test_random_file_matches_oracle_text(tmp_path, k):
    rng = np.random.default_rng(k)
    lengths = np.r_[rng.integers(0, 400, size=400), [30000, 0, 3, 150, 150]]
    fa = tmp_path / "r.fa"
    with open(fa, "wb") as fh:
        for i, n in enumerate(lengths):
            s = bytes(rng.choice(list(b"ACGTNacgtR"), size=int(n), p=[.22, .22, .22, .22, .02, .02, .02, .02, .02, .02]).astype(np.uint8))
            fh.write(b">s%d\n" % i)
            for j in range(0, len(s), 70):
                fh.write(s[j:j + 70] + b"\n")
    out = tmp_path / "o"
    for flags, kw in ((["-k", k], {}), (["-k", k, "-c"], {"norm": False}), (["-k", k, "-r"], {"canonical": False}),
                      (["-k", k, "-r", "-c", "-H", "-p", "csv"], {"canonical": False, "norm": False, "with_header": True, "delim": ","})):
        r = run(["-i", fa, "-o", out, *flags])
        assert r.returncode == 0 and r.stderr == b"", r.stderr
        assert out.read_bytes() == O.comp_oligo_text(fa, k, **kw), flags


def _fasta(path, records, opener=open):
    """records: (name, u8 array); sequences wrapped at 70 columns."""
    with opener(path, "wb") as fh:
        for name, seq in records:
            fh.write(b">" + name + b"\n")
            full = len(seq) // 70
            lines = np.empty((full, 71), dtype=np.uint8)
            lines[:, :70] = seq[:full * 70].reshape(full, 70)
            lines[:, 70] = ord("\n")
            fh.write(lines.tobytes())
            if len(seq) % 70:
                fh.write(seq[full * 70:].tobytes() + b"\n")


def _oversized_seq(rng, n, runs):
    seq = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, size=n, dtype=np.uint8)]
    for _ in range(runs):
        a = int(rng.integers(0, n - 100_000))
        seq[a:a + int(rng.integers(1, 100_000))] = ord("N")
    return seq


OVERSIZED_FLAGS = ((["-k", 4], {}), (["-k", 7, "-c"], {"norm": False}), (["-k", 5, "-r"], {"canonical": False}))


def test_records_larger_than_the_base_buffer(tmp_path):
    """A FASTA file above 32 MiB whose records do not fit the 32 MiB base buffer of a batch: the driver grows the buffer
    set that meets the 36 Mbp record to 1.25 x its size (45 Mbp), and the other set meets a 50 Mbp record after that,
    so both grow, the second from the capacity the first growth set.  The same bytes on stdin, where the buffer starts
    at 32 MiB whatever the input.  Totals above 2^23 also take format_norm_kernel's f64 division."""
    rng = np.random.default_rng(36)

    def short(n):
        return [(b"s%d" % i, _oversized_seq(rng, int(m), 0)) for i, m in enumerate(rng.integers(0, 400, size=n))]

    records = short(5) + [(b"big1", _oversized_seq(rng, 36_000_000, 4))] + short(7) + \
        [(b"big2", _oversized_seq(rng, 50_000_000, 3))] + short(3)
    fa = tmp_path / "big.fa"
    _fasta(fa, records)
    assert fa.stat().st_size > 32 << 20
    data = fa.read_bytes()
    out = tmp_path / "o"
    for flags, kw in OVERSIZED_FLAGS:
        want = O.comp_oligo_text(fa, flags[1], **kw)
        r = run(["-i", fa, "-o", out, *flags])
        assert r.returncode == 0 and r.stderr == b"", r.stderr
        assert out.read_bytes() == want, flags
        r = run(["-i", "-", "-o", out, *flags], stdin=data)
        assert r.returncode == 0 and r.stderr == b"", r.stderr
        assert out.read_bytes() == want, ["stdin", *flags]


def test_gzip_record_far_larger_than_its_file(tmp_path):
    """A 40 Mbp record of a repeated 1 kbp block compresses far below 1/8 of its size, so the base buffer sized from
    the file (8 x its size + 1 MiB) is too small and grows from there."""
    import gzip
    rng = np.random.default_rng(40)
    seq = np.tile(_oversized_seq(rng, 1000, 0), 40_000)
    for a in rng.integers(0, seq.size - 5000, size=4):
        seq[a:a + int(rng.integers(1, 5000))] = ord("N")
    fa = tmp_path / "big.fa.gz"
    _fasta(fa, [(b"s0", seq[:999]), (b"big", seq), (b"s2", seq[5:300])], opener=gzip.open)
    assert fa.stat().st_size * 8 + (1 << 20) < seq.size
    out = tmp_path / "o"
    for flags, kw in OVERSIZED_FLAGS:
        r = run(["-i", fa, "-o", out, *flags])
        assert r.returncode == 0 and r.stderr == b"", r.stderr
        assert out.read_bytes() == O.comp_oligo_text(fa, flags[1], **kw), flags


def test_python_driver_and_many_batches(tmp_path):
    """comp_oligo() through ctypes; enough records for four GPU batches (rows stay in input order), whole output."""
    from kmertools_b200 import io as kio
    rng = np.random.default_rng(2)
    fq = tmp_path / "big.fq"
    n = 3_000
    with open(fq, "wb") as fh:
        arr = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, size=(n, 100))]
        for i in range(n):
            fh.write(b"@r\n" + arr[i].tobytes() + b"\n+\n" + b"I" * 100 + b"\n")
    out, want = tmp_path / "o", tmp_path / "want"
    st = kio.comp_oligo(fq, out, k=7)          # 8192 cols * 9 B = 73.7 kB/row -> 910 rows per 64 MiB batch
    assert st["records"] == n and st["bases"] == n * 100 and st["launches"] >= 8
    O.baseline_text(arr.reshape(-1).copy(), np.arange(n + 1, dtype=np.uint64) * 100, 7, path=str(want))
    assert out.stat().st_size == n * 8192 * 9
    assert out.read_bytes() == want.read_bytes()


def test_comp_cgr_kmer_mode_golden(golden, tmp_path):
    """oligo_cgr_complete_unnorm_test (composition/src/oligocgr.rs:219-238): reads.fq, k=4, vecsize 16, counts."""
    out = tmp_path / "o.cgr"
    r = subprocess.run([str(BIN), "comp", "cgr", "-i", str(golden / "reads.fq"), "-o", str(out), "-k", "4", "-c"],
                       capture_output=True)
    assert r.returncode == 0 and r.stderr == b"", r.stderr
    assert out.read_bytes() == (golden / "expected_reads.k4.cgr").read_bytes()


def test_comp_cgr_normalised_values(golden, tmp_path):
    """Normalised k-mer CGR: freq is Rust's `{}` of the f64 quotient (shortest round-trip digits, never an exponent)."""
    from kmertools_b200 import io as kio
    out = tmp_path / "o.cgr"
    kio.comp_cgr(golden / "reads.fa", out, k=4)
    want = O.comp_cgr_text(golden / "reads.fa", 4, 16)
    assert want.count(b"\n") == 2 and want.startswith(b"(0.5,0.5,")     # AAAA -> (0.5, 0.5), oligocgr.rs:205-206
    assert out.read_bytes() == want
