"""The k-mer pair enumerator (ktb_kmer_pairs / ktb_kmer_pairs_device, csrc/kmer_pairs.cu) where its kernels can go
wrong.  Needs a B200: -m gpu.

pair_count_kernel counts the valid windows of each block of 4096 end positions, pair_scan_kernel (one CTA) scans those
counts in strips of 256 blocks (2^20 bases) and carries the running total from strip to strip, pair_write_kernel stores
every pair at its block's base plus its thread's offset, if that index is below `cap`.  Here: sequences of one, two,
three and six strips with N bytes on strip and block boundaries; device outputs inside sentinel-filled guards at every
capacity, from unaligned `d_seq`; one 4 GiB sequence with more than 2^32 windows and short islands across 2^31 and 2^32;
calls in flight on several streams; and the Python surface.  Every check is integer equality with the CPU oracle."""
import numpy as np
import pytest
import torch

from oracle import oracle as O
from tests.util import assert_rows_equal, random_batch

pytestmark = pytest.mark.gpu

from kmertools_b200 import KmerGenerator, OligoComputer, _lib, kmer_pairs  # noqa: E402
from kmertools_b200._lib import NORM_CLI  # noqa: E402

DEV = torch.device("cuda:0")
# 16 is the last k whose codes fit 32 bits, 17 the first that does not, 31 gives 62-bit codes
KS = [1, 2, 3, 15, 16, 17, 30, 31]
BLOCK = 4096                      # window end positions per CTA (PAIR_THREADS x PAIR_SPAN)
STRIP = 256 * BLOCK               # blocks pair_scan_kernel scans per pass, in bases
P31, P32 = 1 << 31, 1 << 32
GUARD = 4096                      # bytes of guard on each side of d_out_f, d_out_r and d_count
SENTINEL = 0x7FF8DEAD0BADF00D     # over 2^62: no pair code and no count equals it
N = ord("N")
# bases in every spelling kmer.rs:6-15 accepts: upper and lower case, U, raw 0..3 codes
MIXED = np.frombuffer(b"ACGTacgtUu\x00\x01\x02\x03", dtype=np.uint8)


def mixed(rng, n):
    return MIXED[rng.integers(0, len(MIXED), size=n)]


def _stream(s):
    return None if s is None else s.cuda_stream


def assert_pairs(f, r, want, what):
    wf, wr, wm = want
    assert len(f) == len(r) == wm, f"{what}: {len(f)} / {len(r)} pairs, want {wm}"
    for name, got, w in (("forward", f, wf), ("reverse", r, wr)):
        got = np.asarray(got, dtype=np.uint64)
        if not np.array_equal(got, w):
            i = int(np.flatnonzero(got != w)[0])
            raise AssertionError(f"{what}: {name} codes differ, first at pair {i}: got {int(got[i]):#x} want {int(w[i]):#x}")


# ---------------------------------------------------------------------------------------------------------------------
# fenced device outputs

class Fence:
    """d_out_f and d_out_r (`cap` elements) and d_count, each inside an int64 buffer with GUARD bytes of guard on either
    side, all preset to SENTINEL.  With cap = 0 the outputs are passed as NULL."""

    def __init__(self, cap):
        g = GUARD // 8
        self.cap = cap
        self.f = torch.full((2 * g + cap,), SENTINEL, dtype=torch.int64, device=DEV)
        self.r = torch.full((2 * g + cap,), SENTINEL, dtype=torch.int64, device=DEV)
        self.n = torch.full((2 * g + 1,), SENTINEL, dtype=torch.int64, device=DEV)
        self.f_ptr = self.f.data_ptr() + GUARD if cap else None
        self.r_ptr = self.r.data_ptr() + GUARD if cap else None

    def enqueue(self, d_seq, n, k, stream):
        """One ktb_kmer_pairs_device call on `stream` (a torch stream, or None for the legacy default stream)."""
        _lib.check(_lib.load().ktb_kmer_pairs_device(d_seq, n, k, self.f_ptr, self.r_ptr, self.cap,
                                                     self.n.data_ptr() + GUARD, _stream(stream)))

    def check(self, want, what):
        """Guards unchanged, *d_count = the oracle count, the first min(count, cap) pairs = the oracle's, every element
        from min(count, cap) on still the sentinel.  `want` = (f, r, count); f and r need only min(count, cap) pairs."""
        g = GUARD // 8
        bufs = {name: t.cpu().numpy().view(np.uint64) for name, t in (("d_out_f", self.f), ("d_out_r", self.r),
                                                                      ("d_count", self.n))}
        for name, b in bufs.items():
            for side, part in (("before", b[:g]), ("after", b[len(b) - g:])):
                bad = np.flatnonzero(part != SENTINEL)
                assert bad.size == 0, f"{what}: {bad.size} words of the guard {side} {name} changed, first at word " \
                                      f"{int(bad[0])} of it"
        wf, wr, wm = want
        count = int(bufs["d_count"][g])
        assert count == wm, f"{what}: *d_count = {count:#x}, want {wm:#x}"
        m = min(count, self.cap)
        for name, w in (("d_out_f", wf), ("d_out_r", wr)):
            body = bufs[name][g:g + self.cap]
            if m and not np.array_equal(body[:m], w[:m]):
                i = int(np.flatnonzero(body[:m] != w[:m])[0])
                raise AssertionError(f"{what}: {name} differs, first at pair {i} of {m}: got {int(body[i]):#x} "
                                     f"want {int(w[i]):#x}")
            wrote = np.flatnonzero(body[m:] != SENTINEL)
            assert wrote.size == 0, f"{what}: {name} written at {wrote.size} elements at or beyond min(count, cap) = " \
                                    f"{m}, first at {m + int(wrote[0])}"


def resident(seq, offset=0):
    """(tensor, d_seq) with `seq` at byte `offset` of a device tensor.  ACGT bytes sit before it and 64 after it, so a
    read outside [d_seq, d_seq + len) adds or changes pairs."""
    fill = np.frombuffer(b"ACGT" * (offset // 4 + 17), dtype=np.uint8)
    t = torch.from_numpy(np.concatenate([fill[:offset], seq, fill[:64]])).to(DEV)
    return t, t.data_ptr() + offset


@pytest.fixture(scope="module", autouse=True)
def _release():
    yield
    _drop_big()


# ---------------------------------------------------------------------------------------------------------------------
# the scan past its first strip, through the host entry point

def with_boundary_ns(rng, seq):
    """N bytes and short N runs on every strip boundary (p = m * 2^20 - 1 or m * 2^20) and on a quarter of the block
    boundaries (p = b * 4096 - 1 or b * 4096); windows cross every other boundary."""
    n = len(seq)
    for m in range(1, (n - 1) // STRIP + 1):
        p = m * STRIP
        kind = m % 3
        if kind == 0:
            seq[p - 1] = N
        elif kind == 1:
            seq[p] = N
        else:
            seq[p - int(rng.integers(1, 4)):p + int(rng.integers(1, 4))] = N
    for b in range(1, (n - 1) // BLOCK + 1):
        p, u = b * BLOCK, rng.random()
        if p % STRIP == 0 or u >= 0.25:
            continue
        if u < 0.1:
            seq[p - 1] = N
        elif u < 0.2:
            seq[p] = N
        else:
            seq[p - int(rng.integers(0, 6)):p + int(rng.integers(1, 6))] = N
    return seq


STRIP_LENGTHS = [STRIP - 1, STRIP, STRIP + 1, STRIP + 256 * BLOCK + 15, 5 * STRIP + 3]
_strip_seqs = {}


def strip_seq(n):
    if n not in _strip_seqs:
        rng = np.random.default_rng(n)
        _strip_seqs[n] = with_boundary_ns(rng, mixed(rng, n))
    return _strip_seqs[n]


@pytest.mark.parametrize("n", STRIP_LENGTHS, ids=lambda n: f"{n // BLOCK}blocks+{n % BLOCK}")
@pytest.mark.parametrize("k", KS)
def test_scan_strips_host_entry(k, n):
    """2^20 - 1 and 2^20 bases fill one strip of the scan, 2^20 + 1 starts a second, 2^21 + 15 ends in a third strip of
    one block, 5 * 2^20 + 3 carries the running total five times."""
    seq = strip_seq(n)
    f, r = kmer_pairs(seq, k)
    assert_pairs(f, r, O.kmer_arrays(seq, k), f"n={n} k={k}")


def test_scan_40_mbp_k31():
    """One 40 Mbp sequence (39 strips) with noise bytes, an N run and N bytes on the strip and block boundaries."""
    rng = np.random.default_rng(40)
    n = 40_000_000
    bases, _ = random_batch(rng, [n], noise=0.01, n_runs=1.0)
    seq = with_boundary_ns(rng, bases)
    f, r = kmer_pairs(seq, 31)
    want = O.kmer_arrays(seq, 31)
    assert want[2] > n // 2
    assert_pairs(f, r, want, "40 Mbp k=31")


# ---------------------------------------------------------------------------------------------------------------------
# fenced device outputs at every capacity, from unaligned d_seq

def fenced_cases(k):
    """(name, sequence, cap): a 60 kbp sequence with N bytes at cap > count, cap = count, cap cutting a block and a
    thread span in the middle, and cap = 0 with NULL outputs; then len = 0, 0 < len < k and len = k."""
    rng = np.random.default_rng(600 + k)
    seq = mixed(rng, 60_000)
    seq[rng.random(seq.size) < 0.002] = N
    seq[20_000:20_100] = N
    count = O.kmer_arrays(seq, k, want_pairs=False)
    assert count > 3 * BLOCK + 7 + 10_000
    cases = [("cap > count", seq, count + 37), ("cap = count", seq, count), ("cap mid-span", seq, 3 * BLOCK + 7),
             ("count only", seq, 0), ("len = 0", seq[:0], 8)]
    if k > 1:
        cases.append(("0 < len < k", mixed(rng, k - 1), 8))
    cases.append(("len = k", mixed(rng, k), 8))
    return cases


@pytest.mark.parametrize("offset", [0, 1, 7, 15])
@pytest.mark.parametrize("k", KS)
def test_fenced_device_outputs(k, offset):
    """Nothing at or beyond min(count, cap) is written, nothing outside the outputs, and d_seq needs no alignment."""
    stream = torch.cuda.current_stream()
    for name, seq, cap in fenced_cases(k):
        t, d_seq = resident(seq, offset)
        fence = Fence(cap)
        fence.enqueue(d_seq if seq.size else None, seq.size, k, stream)
        stream.synchronize()
        fence.check(O.kmer_arrays(seq, k), f"{name} (len {seq.size}, cap {cap}) k={k} offset={offset}")


# ---------------------------------------------------------------------------------------------------------------------
# positions, block bases and counts past 2^31 and 2^32

BIG = P32 + 3 * BLOCK + 37        # 2^20 + 4 blocks, the last one 37 bases: a partial thread span in a partial block
_big = {}


def _drop_big():
    _big.clear()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


def islands(rng):
    """(start, bytes) of short runs of bases in an N-filled buffer, each separated from the next by N bytes."""
    spans = [(0, 50), (P31 - 40, P31 + 40), (P32 - 33, P32 + 47), (P32 + BLOCK - 20, P32 + BLOCK + 20), (BIG - 60, BIG)]
    return [(a, mixed(rng, b - a)) for a, b in spans]


ISLANDS = islands(np.random.default_rng(32))


def big(fill):
    """The module's one BIG-byte device buffer, filled with `fill`:
      "random"  : random raw codes 0..3 (every window valid).  Random, not a repeat: with a periodic pattern a pair
                  written to an index wrapped by 2^32 would hold the right value by accident.
      "islands" : N everywhere except ISLANDS."""
    if "buf" not in _big:
        _big["buf"] = torch.empty(BIG, dtype=torch.uint8, device=DEV)
    buf = _big["buf"]
    if _big.get("fill") != fill:
        if fill == "random":
            buf.random_(0, 4, generator=torch.Generator(device=DEV).manual_seed(2024))
        else:
            buf.fill_(N)
            for a, s in ISLANDS:
                buf[a:a + s.size].copy_(torch.from_numpy(s))
        _big["fill"] = fill
    return buf


def islands_want(k):
    parts = [O.kmer_arrays(s, k) for _, s in ISLANDS]
    return np.concatenate([p[0] for p in parts]), np.concatenate([p[1] for p in parts]), sum(p[2] for p in parts)


def test_host_entry_past_2_31():
    """ktb_kmer_pairs on a host buffer of 2^31 + 3 * 4096 + 11 bytes, N but for islands at the start, across 2^31 and at
    the end; a small cap, so the outputs are not 16 bytes per base."""
    import ctypes as C
    _drop_big()   # this call copies the sequence to a device buffer of its own
    n = P31 + 3 * BLOCK + 11
    host = np.full(n, N, dtype=np.uint8)
    rng = np.random.default_rng(31)
    parts = [(0, mixed(rng, 40)), (P31 - 40, mixed(rng, 80)), (n - 45, mixed(rng, 45))]
    for a, s in parts:
        host[a:a + s.size] = s
    for k in (1, 17, 31):
        want = [O.kmer_arrays(s, k) for _, s in parts]
        wm = sum(w[2] for w in want)
        cap = wm + 64
        f = np.full(cap, SENTINEL, dtype=np.uint64)
        r = np.full(cap, SENTINEL, dtype=np.uint64)
        count = C.c_uint64()
        _lib.check(_lib.load().ktb_kmer_pairs(host.ctypes.data, n, k, 0, f.ctypes.data, r.ctypes.data, cap,
                                              C.byref(count)))
        assert count.value == wm, (k, count.value, wm)
        assert_pairs(f[:wm], r[:wm], (np.concatenate([w[0] for w in want]), np.concatenate([w[1] for w in want]), wm),
                     f"host 2^31 k={k}")
        assert (f[wm:] == SENTINEL).all() and (r[wm:] == SENTINEL).all(), f"k={k}: written beyond the count"


@pytest.mark.parametrize("k", [1, 17, 31])
def test_more_than_2_32_windows(k):
    """L - k + 1 > 2^32 valid windows: the count must not wrap, and no block's output index may wrap into the first
    cap = 2^20 + 5 pairs."""
    buf = big("random")
    total = BIG - k + 1
    assert total > P32
    stream = torch.cuda.current_stream()
    fence = Fence(0)
    fence.enqueue(buf.data_ptr(), BIG, k, stream)
    stream.synchronize()
    fence.check((None, None, total), f"count only k={k}")
    cap = STRIP + 5
    head = buf[:cap + k - 1].cpu().numpy()
    assert head.max() < 4 and np.bincount(head, minlength=4).min() > cap // 5
    wf, wr, wm = O.kmer_arrays(head, k)
    assert wm == cap
    fence = Fence(cap)
    fence.enqueue(buf.data_ptr(), BIG, k, stream)
    stream.synchronize()
    fence.check((wf, wr, total), f"cap {cap} k={k}")


@pytest.mark.parametrize("k", KS)
def test_islands_past_2_31_and_2_32(k):
    """Islands at the start, across 2^31, across 2^32, across the block boundary 2^32 + 4096 and in the last 60 bytes
    (a partial thread span of the partial last block): their pairs, in order, with cap = count and with cap = 0."""
    buf = big("islands")
    want = islands_want(k)
    assert want[2] > 0
    stream = torch.cuda.current_stream()
    for cap in (want[2], 0):
        fence = Fence(cap)
        fence.enqueue(buf.data_ptr(), BIG, k, stream)
        stream.synchronize()
        fence.check(want, f"islands cap {cap} k={k}")


# ---------------------------------------------------------------------------------------------------------------------
# calls in flight together

def _flight_seq(rng, n):
    seq = mixed(rng, n)
    seq[rng.random(n) < 0.003] = N
    return seq


def _enqueue_job(seq, calls, stream, pending, what):
    """calls: (k, cap) enqueued back to back on `stream` with no host sync; cap None = every pair, "half" = about half
    of them (a cut inside a block).  The sequence and the fences are written on `stream` too."""
    wants = [O.kmer_arrays(seq, k) for k, _ in calls]
    with torch.cuda.stream(stream if stream is not None else torch.cuda.default_stream(DEV)):
        t, d_seq = resident(seq, 3)
        for (k, cap), want in zip(calls, wants):
            c = {None: want[2], "half": want[2] // 2 + 7}.get(cap, cap)
            fence = Fence(c)
            fence.enqueue(d_seq, seq.size, k, stream)
            pending.append((fence, want, f"{what} k={k} cap={c}", t))


def test_calls_in_flight_on_four_streams():
    """Three streams enqueue two enumerator calls each (own sequence, k and fences), a fourth runs vectorise_tensors,
    all before one synchronize.  Every call takes its scratch from the stream-ordered allocator of its own stream."""
    rng = np.random.default_rng(77)
    jobs = [(_flight_seq(rng, 1_500_000), [(31, None), (31, "half")]),
            (_flight_seq(rng, 300_001), [(16, "half"), (16, 0)]),
            (_flight_seq(rng, 70_000), [(1, None), (1, 5)])]
    bases, offsets = random_batch(rng, np.r_[rng.integers(100, 251, size=64), [200_000, 0, 6, 4096]], noise=0.01)
    want_rows = O.vectorise_batch(bases, offsets, 7, True, NORM_CLI)[0]
    oc = OligoComputer(7)
    pending = []
    streams = [torch.cuda.Stream(device=DEV) for _ in range(4)]
    for (seq, calls), s in zip(jobs, streams):
        _enqueue_job(seq, calls, s, pending, f"stream job of {seq.size} bases")
    with torch.cuda.stream(streams[3]):
        d_bases = torch.from_numpy(bases).to(DEV)
        d_offsets = torch.from_numpy(offsets.astype(np.int64)).to(DEV)
        rows = oc.vectorise_tensors(d_bases, d_offsets, norm_mode=NORM_CLI, mins=True, dtype=torch.float32)
    torch.cuda.synchronize()
    for fence, want, what, _ in pending:
        fence.check(want, what)
    assert_rows_equal(rows.cpu().numpy(), want_rows, np.float32, "vectorise_tensors beside the enumerator")
    oc.close()


def test_calls_in_flight_on_the_legacy_default_stream():
    rng = np.random.default_rng(78)
    pending = []
    _enqueue_job(_flight_seq(rng, 1_100_000), [(17, None), (3, "half"), (30, 0)], None, pending, "default stream")
    _enqueue_job(_flight_seq(rng, 9_000), [(2, None)], None, pending, "default stream, small")
    torch.cuda.synchronize()
    for fence, want, what, _ in pending:
        fence.check(want, what)


# ---------------------------------------------------------------------------------------------------------------------
# the Python surface

def test_kmer_pairs_input_types():
    """str, bytes, bytearray, memoryview, a uint8 array and a strided view all enumerate the same bytes."""
    rng = np.random.default_rng(90)
    arr = _flight_seq(rng, 10_000)
    b = arr.tobytes()
    spread = np.frombuffer(b"ACGT" * (arr.size // 2), dtype=np.uint8).copy()   # arr in its even bytes, bases between
    spread[::2] = arr
    view = spread[::2]
    assert not view.flags.c_contiguous
    for k in KS:
        want = O.kmer_arrays(arr, k)
        for name, x in (("str", b.decode("ascii")), ("bytes", b), ("bytearray", bytearray(b)), ("memoryview",
                        memoryview(b)), ("array", arr), ("strided view", view)):
            assert_pairs(*kmer_pairs(x, k), want, f"{name} k={k}")


def test_non_ascii_str_and_generator():
    """A str is enumerated as its UTF-8 bytes (bytes >= 128 are not bases); KmerGenerator yields the same pairs."""
    s = ("ACGTTGCAé" + "ACGT" * 9 + "漢字acgtu" + "GATTACA" * 6 + "𝄞\x00\x01\x02\x03ACGTN") * 40
    raw = s.encode("utf-8")
    assert max(raw) >= 128
    for k in KS:
        want = O.kmer_arrays(raw, k)
        assert want[2] > 0
        assert_pairs(*kmer_pairs(s, k), want, f"non-ASCII str k={k}")
        assert list(KmerGenerator(s, k)) == O.kmers(raw, k), f"KmerGenerator k={k}"


@pytest.mark.parametrize("k", range(1, 13))
def test_kmer_pos_maps_every_k(k):
    pos_map, pos_to_kmer, count = KmerGenerator("", k).kmer_pos_maps()
    om, ok, oc = O.kmer_pos_maps(k)
    assert count == oc == len(pos_to_kmer) and len(pos_map) == 4 ** k
    assert np.array_equal(np.asarray(pos_map, dtype=np.uint64), om)
    assert np.array_equal(np.fromiter((pos_to_kmer[j] for j in range(count)), dtype=np.uint64, count=count), ok)


def test_kmer_pos_maps_k13_raises():
    with pytest.raises(ValueError):
        KmerGenerator("", 13).kmer_pos_maps()


def test_second_device():
    if _lib.load().ktb_device_count() < 2:
        pytest.skip("needs two GPUs")
    torch.cuda.set_device(0)
    rng = np.random.default_rng(91)
    seq = _flight_seq(rng, 1_200_000)
    for k in (1, 17, 31):
        assert_pairs(*kmer_pairs(seq, k, device=1), O.kmer_arrays(seq, k), f"device 1 k={k}")
        assert torch.cuda.current_device() == 0
