"""Pins the CPU oracle against every golden vector / KAT the reference holds for the oligo path.

Reference tests restated here: kmer/src/kmer.rs:113-176, kmer/src/lib.rs:56-71,
composition/src/oligo.rs:269-432, composition/src/oligocgr.rs:199-208, tests/test_oligo.py:8-35.
"""
import hashlib

import numpy as np
import pytest

from oracle import oracle as O


def test_nt4_table():
    valid = {0: 0, 1: 1, 2: 2, 3: 3, ord("A"): 0, ord("a"): 0, ord("C"): 1, ord("c"): 1,
             ord("G"): 2, ord("g"): 2, ord("T"): 3, ord("t"): 3, ord("U"): 3, ord("u"): 3}
    for b in range(256):
        assert O.nt4(b) == valid.get(b, 4)


def test_kmers_generated():  # kmer.rs:113-128
    assert O.kmers(b"ACGT", 2) == [(1, 11), (6, 6), (11, 1)]


def test_kmers_generated_ambiguous():  # kmer.rs:130-145
    assert O.kmers(b"ACNGTT", 2) == [(1, 11), (11, 1), (15, 0)]


def test_kmer_arrays_match_kmers():
    """kmer_arrays (uint64 arrays, what the large GPU tests compare with) == kmers (tuples) on short sequences."""
    rng = np.random.default_rng(11)
    mixed = np.frombuffer(b"ACGTacgtUuNR\x00\x01\x02\x03\xc3\xa9", dtype=np.uint8)
    seqs = [b"", b"A", b"ACGT", b"ACNGTT", b"NNNN", bytes(range(256)) * 2]
    seqs += [mixed[rng.integers(0, len(mixed), size=n)].tobytes() for n in (5, 31, 32, 100, 777)]
    for seq in seqs:
        for k in (1, 2, 3, 15, 16, 17, 30, 31):
            want = O.kmers(seq, k)
            for buf in (seq, np.frombuffer(seq, dtype=np.uint8)):
                f, r, m = O.kmer_arrays(buf, k)
                assert f.dtype == r.dtype == np.uint64 and m == len(f) == len(r) == len(want), (seq[:16], k)
                assert list(zip(f.tolist(), r.tolist())) == want, (seq[:16], k)
                assert O.kmer_arrays(buf, k, want_pairs=False) == m
    arr = np.frombuffer(b"ACGTTGCAACGTAGCT" * 4, dtype=np.uint8)
    f, r, m = O.kmer_arrays(arr[::3], 5)   # a strided view is read as the bytes it shows
    assert list(zip(f.tolist(), r.tolist())) == O.kmers(arr[::3].tobytes(), 5) and m > 0


def test_rev_comp():  # kmer.rs:147-153
    assert O.rev_comp(0b00011011, 4) == 0b00011011
    assert O.rev_comp(0b001101101011, 6) == 0b000101100011


def test_pos_map():  # kmer.rs:155-176
    pos_map, p2k, cnt = O.kmer_pos_maps(4)
    assert cnt == 136 and len(p2k) == 136
    assert int((pos_map > 0).sum()) == 135
    assert pos_map.max() < 136
    assert pos_map[0] == 0 and pos_map[0xFF] == 0 and pos_map[3] == 3


@pytest.mark.parametrize("k,d", [(1, 2), (2, 10), (3, 32), (4, 136), (5, 512), (6, 2080), (7, 8192),
                                 (8, 32896), (9, 131072), (10, 524800)])
def test_dims(k, d):
    assert O.dim(k, True) == d
    assert O.dim(k, False) == 4 ** k


def test_numeric_kmer_roundtrip():  # kmer/src/lib.rs:56-71
    assert O.numeric_to_kmer(0b0001101111, 5) == "ACGTT"
    assert O.kmer_to_numeric("ACGTT") == (111, 27)


def test_kmer_vec_unit_kats():  # composition/src/oligo.rs:269-309
    raw = O.vectorise_one(b"AAAANGAGA", 4, canonical=False, norm_mode=0)
    assert len(raw) == 256
    v = O.vectorise_one(b"AAAANGAGA", 4, canonical=True, norm_mode=1)
    assert v[0] == 0.5
    u = O.vectorise_one(b"AAAANGAGA", 4, canonical=True, norm_mode=0)
    assert u[0] == 1.0 and u.sum() == 2.0


def test_header():  # composition/src/oligo.rs:389-400, tests/test_oligo.py:28-35
    h = O.header(4, True)
    assert len(h) == 136 and h[0] == "AAAA" and h[135] == "TTAA"
    hr = O.header(4, False)
    assert len(hr) == 256 and hr[0] == "AAAA" and hr[255] == "TTTT"


def test_lowercase_kat():  # composition/src/oligocgr.rs:199-208: "aaaatg..." k=4 -> 1/26 in slot 0
    seq = b"aaaatgatgaaatagagagactttattaa"
    v = O.vectorise_one(seq, 4)
    assert v[0] == 1.0 / (29 - 4 + 1)
    assert O.vectorise_one(seq.upper(), 4).tolist() == v.tolist()


@pytest.mark.parametrize("fname", ["reads.fa", "reads.fq", "reads.fq.gz"])
def test_golden_norm(golden, fname):  # vec_mmap_test / vec_batch_threaded_test
    assert O.comp_oligo_text(golden / fname, 4) == (golden / "expected_fa.kmers").read_bytes()


def test_golden_unnorm(golden):  # vec_batch_threaded_unnorm_test
    got = O.comp_oligo_text(golden / "reads.fa", 4, norm=False)
    assert got == (golden / "expected_fa_batch_unnorm.kmers").read_bytes()


def test_golden_header(golden):  # vec_batch_with_header_test / vec_mmap_with_header_test
    got = O.comp_oligo_text(golden / "reads.fa", 4, with_header=True)
    assert got == (golden / "expected_fa_header.kmers").read_bytes()


def test_cgr_text_golden(golden):  # oligo_cgr_complete_unnorm_test, composition/src/oligocgr.rs:219-238
    assert O.comp_cgr_text(golden / "reads.fq", 4, 16, norm=False) == (golden / "expected_reads.k4.cgr").read_bytes()
    assert O.cgr_points(4, 16)[0] == (0.5, 0.5)   # AAAA, oligocgr.rs:205-206
    # Rust's `{}` never switches to an exponent and drops a trailing ".0"
    for v, want in ((0.0, "0"), (1.0, "1"), (8.5, "8.5"), (1 / 3, "0.3333333333333333"), (1e-7, "0.0000001"),
                    (1 / 16777219, "0.000000059604634117251494"), (123456.0, "123456")):
        assert O._rust_f64(v) == want


def test_python_binding_golden(golden):  # tests/test_oligo.py:8-25
    seqs = [s for _, s in O.read_fastx(golden / "reads.fq")]
    bases, offsets = O.pack(seqs)
    rows, _ = O.vectorise_batch(bases, offsets, 4, True, 2)
    truth = [list(map(float, ln.split())) for ln in (golden / "expected_fa.kmers").read_text().splitlines()]
    assert [[round(x, 6) for x in r] for r in rows.tolist()] == truth


def test_seq_reader(golden):  # ktio/src/seq.rs:164-233
    for f in ["reads.fa", "reads.fq", "reads.fq.gz"]:
        recs = O.read_fastx(golden / f)
        want = ["Record_1", "Record_2"] if f.endswith(".fa") else ["Read_1", "Read_2"]
        assert [r[0] for r in recs] == want
        assert sum(len(r[1]) for r in recs) == 144
    assert O.read_fastx(golden / "reads.fa")[0][1] == \
        b"GGGTGATGGCCGCTGCCGATGGCGTCAAATCCCACCAAGTTACCCTTAACAACTTAAGGGTTTTCAAATAGA"


# sha256[:16] of comp-oligo text on reads.fa, from SURVEY.md §8c (independent restatement made during
# the survey): k -> (canonical-norm, canonical-counts, raw-norm, raw-counts)
SURVEY_KATS = {
    3: ("7f4303e48b69b801", "fe762ced23d632ab", "f89f59a56f353aa1", "4697a1a984e00ab7"),
    4: ("981027c2e3823baf", "6c77f37ca0baf48e", "9ce44b73a355df20", "af7ac36b1c297d44"),
    5: ("09743a02344004ea", "bebb1221fc48cf4e", "c4d2716114da8b49", "d05058a8bddcbb14"),
    6: ("b4ca0e00c6c659c8", "26c07a42b3d7574e", "b1976e8c858332c2", "c73b075ad53ffe40"),
    7: ("abc83d10708c3201", "be71e3a4747092da", "e493b2fae10fe843", "44d0f7b6fa2ffb8c"),
}


@pytest.mark.parametrize("k", sorted(SURVEY_KATS))
def test_survey_derived_hashes(golden, k):
    want = SURVEY_KATS[k]
    got = []
    for canonical in (True, False):
        for norm in (True, False):
            txt = O.comp_oligo_text(golden / "reads.fa", k, canonical=canonical, norm=norm)
            got.append(hashlib.sha256(txt).hexdigest()[:16])
    assert tuple(got) == want


def test_edge_cases():  # SURVEY.md §8c
    for s in (b"ACG", b"", b"NNNNNNNN"):
        assert not O.vectorise_one(s, 4).any()
    a = O.vectorise_one(b"acgu", 4, norm_mode=0)
    assert a.tolist() == O.vectorise_one(b"ACGT", 4, norm_mode=0).tolist()
    assert a.tolist() == O.vectorise_one(bytes([0, 1, 2, 3]), 4, norm_mode=0).tolist()
    assert a[27] == 1 and a.sum() == 1
    assert O.vectorise_one(b"ACGTRACGT", 4, norm_mode=0).sum() == 2


def test_py_raw_quirk():  # pybindings/src/oligo.rs:58-62 — raw normalised vectors sum to 0.5
    seq = b"ACGTTGCAACGTAGCTAGCTAGGATCGA"
    assert O.vectorise_one(seq, 3, canonical=False, norm_mode=2).sum() == pytest.approx(0.5)
    assert O.vectorise_one(seq, 3, canonical=False, norm_mode=1).sum() == pytest.approx(1.0)
    assert O.vectorise_one(seq, 3, canonical=True, norm_mode=2).sum() == pytest.approx(1.0)


def test_closed_form_matches_state_machine():
    """SURVEY §8a closed form (what the GPU kernels implement) == the serial iterator."""
    rng = np.random.default_rng(7)
    alphabet = np.frombuffer(b"ACGTacgtNRYKM-\x00\x01\x02\x03Uu", dtype=np.uint8)
    for k in (1, 2, 3, 5, 8, 13, 31):
        for _ in range(20):
            L = int(rng.integers(0, 80))
            p = np.r_[np.full(8, 0.1), np.full(len(alphabet) - 8, 0.2 / (len(alphabet) - 8))]
            seq = rng.choice(alphabet, size=L, p=p / p.sum()).astype(np.uint8).tobytes()
            code = [O.nt4(b) for b in seq]
            want = []
            for e in range(k - 1, L):
                win = code[e - k + 1:e + 1]
                if all(c < 4 for c in win):
                    f = 0
                    r = 0
                    for j, c in enumerate(win):
                        f |= c << (2 * (k - 1 - j))
                        r |= (3 - c) << (2 * j)
                    want.append((f, r))
            assert O.kmers(seq, k) == want
