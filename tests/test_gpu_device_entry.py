"""The device entry point (ktb_oligo_vectorise_device) as a caller that keeps its batches on the GPU uses it.  Needs a
B200: -m gpu.

The host entry point reshapes every batch before a kernel sees it: offsets rebased to the chunk, at most 2^30 bases per
chunk, rows in a library buffer, one call at a time.  A torch caller gets none of that: its batch may sit anywhere in a
large resident buffer (base positions past 2^31 and 2^32, `offsets[0]` far from 0), its rows land in a caching allocator
next to other tensors, and it enqueues several calls before it synchronises.  Every call here writes into fenced
buffers (sentinels inside, guards around) and is compared bit for bit with the f64 oracle."""
import numpy as np
import pytest
import torch

from oracle import oracle as O
from tests.test_gpu_large_sequences import PATHS, _id
from tests.test_gpu_parity import OPTION_DEFAULTS
from tests.util import ALPHA, assert_rows_equal, random_batch

pytestmark = pytest.mark.gpu

from kmertools_b200 import OligoComputer  # noqa: E402
from kmertools_b200._lib import NORM_CLI, NORM_COUNTS, NORM_PY, OUT_F32, OUT_F64, OUT_U32  # noqa: E402

DEV = torch.device("cuda:0")
CODE = {np.dtype(np.uint32): OUT_U32, np.dtype(np.float32): OUT_F32, np.dtype(np.float64): OUT_F64}
GUARD = 4096                                          # bytes of guard on each side of the rows and of the totals
SENTINEL = {4: 0x7FC0DEAD, 8: 0x7FF8DEAD0BADF00D}     # quiet NaNs that are no plausible count either
_WORD = {4: torch.int32, 8: torch.int64}

_handles = {}


def handle(k, tag=0):
    """Handles of this module, closed at its end (the bucket path sizes its scratch by total_bases, which is 2^32 here)."""
    if (k, tag) not in _handles:
        _handles[(k, tag)] = OligoComputer(k)
    return _handles[(k, tag)]


@pytest.fixture(scope="module", autouse=True)
def _release():
    yield
    global _big
    _big = None
    for oc in _handles.values():
        oc.close()
    _handles.clear()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


def _acgt(rng, n):
    return ALPHA[rng.integers(0, 4, size=n, dtype=np.uint8)]


def _seq(rng, n, noise=0.0, n_runs=0.0):
    return random_batch(rng, [n], noise=noise, n_runs=n_runs)[0]


# ---------------------------------------------------------------------------------------------------------------------
# batches: host bytes (rebased to 0) for the oracle, and where they live on the device

class Batch:
    """`bases`/`offsets` on the host from 0; `buf` is the device buffer whose start is d_bases, `d_offsets` the absolute
    offsets into it (offsets + `at`)."""

    def __init__(self, name, bases, offsets, buf, at):
        self.name, self.bases, self.offsets, self.buf, self.at = name, bases, offsets, buf, at
        self.n = len(offsets) - 1
        self.d_offsets = torch.from_numpy(offsets.astype(np.int64) + at).to(DEV)
        self.total = int(offsets[-1]) + at    # total_bases = offsets[n], as the header requires


def pack(members):
    lengths = [len(m) for m in members]
    offsets = np.zeros(len(members) + 1, dtype=np.uint64)
    np.cumsum(lengths, out=offsets[1:])
    bases = np.concatenate(members) if members else np.zeros(0, np.uint8)
    return bases, offsets


def resident(name, members, at=0):
    """A device buffer holding ACGT filler, the batch at byte `at`, and 64 more filler bytes behind it."""
    bases, offsets = pack(members)
    fill = np.frombuffer(b"ACGT" * ((at + 64) // 4 + 1), np.uint8)
    host = np.concatenate([fill[:at], bases, fill[:64]])
    return Batch(name, bases, offsets, torch.from_numpy(host).to(DEV), at)


_oracle = {}


def oracle(b, k, mins, norm):
    """Oracle rows and totals, once per (batch, k, canonical, norm mode); one k is cached at a time."""
    key = (b.name, k, mins, norm)
    if key not in _oracle:
        if any(kk != k for _, kk, _, _ in _oracle):
            _oracle.clear()
        _oracle[key] = O.vectorise_batch(b.bases, b.offsets, k, mins, norm)
    return _oracle[key]


# ---------------------------------------------------------------------------------------------------------------------
# fenced outputs

class Fence:
    """Rows (n x dim) and totals (n) inside larger buffers, GUARD bytes of guard on each side, everything preset to a
    sentinel (rows, guards) or -1 (totals).  check() finds guards that changed, elements no kernel wrote, and rows or
    totals that differ from the oracle."""

    def __init__(self, n, dim, dtype, with_totals):
        self.n, self.dim, self.dtype = n, dim, np.dtype(dtype)
        es = self.dtype.itemsize
        self.g, self.s = GUARD // es, SENTINEL[es]
        self.rows = torch.full((2 * self.g + n * dim,), self.s, dtype=_WORD[es], device=DEV)
        self.tot = torch.full((2 * (GUARD // 8) + n,), -1, dtype=torch.int64, device=DEV) if with_totals else None
        self.out_ptr = self.rows.data_ptr() + GUARD
        self.tot_ptr = self.tot.data_ptr() + GUARD if with_totals else None

    @staticmethod
    def _fenced(buf, g, count, s, what):
        head, body, tail = buf[:g], buf[g:g + count], buf[g + count:]
        for side, part in (("before", head), ("after", tail)):
            bad = torch.nonzero(part != s)
            assert bad.numel() == 0, f"{what}: {bad.numel()} words of the guard {side} the output changed, " \
                                     f"first at word {int(bad[0])} of it"
        left = torch.nonzero(body == s)
        assert left.numel() == 0, f"{what}: {left.numel()} elements never written, first at element {int(left[0])}"
        return body

    def check(self, want, wtot, what):
        body = self._fenced(self.rows, self.g, self.n * self.dim, self.s, f"{what} rows")
        got = body.cpu().numpy().view(self.dtype).reshape(self.n, self.dim)
        assert_rows_equal(got, want, self.dtype, what)
        if self.tot is not None:
            t = self._fenced(self.tot, GUARD // 8, self.n, -1, f"{what} totals")
            assert np.array_equal(t.cpu().numpy().astype(np.uint64), wtot), f"{what}: totals differ"


def set_options(oc, opts):
    assert set(opts) <= {key for key, _ in OPTION_DEFAULTS}, opts
    for key, dflt in OPTION_DEFAULTS:
        oc.set_option(key, opts.get(key, dflt))


def enqueue(oc, b, mins, norm, dtype, *, stream, totals=True, opts=None):
    """One device call on `stream` (a torch stream, or None for the legacy default stream) into a fresh Fence; options
    apply to this call only."""
    fence = Fence(b.n, oc.dim(mins), dtype, totals)
    set_options(oc, opts or {})
    try:
        oc.vectorise_device(b.buf.data_ptr(), b.d_offsets.data_ptr(), b.n, b.total, fence.out_ptr, norm_mode=norm,
                            mins=mins, out_dtype=CODE[np.dtype(dtype)], d_totals=fence.tot_ptr,
                            stream=None if stream is None else stream.cuda_stream)
    finally:
        set_options(oc, {})
    return fence


def checked_call(k, b, mins, norm, dtype, what, *, totals=True, opts=None):
    stream = torch.cuda.current_stream()
    fence = enqueue(handle(k), b, mins, norm, dtype, stream=stream, totals=totals, opts=opts)
    stream.synchronize()
    fence.check(*oracle(b, k, mins, norm), what)


def pinned(k, mins, opts):
    """The options of a PATHS entry with every heuristic choice it relies on made explicit.  The heuristics read the
    mean length as total_bases / n, which is 2^32 / n at the high offsets and a few kbp in the edge batch.

    With these pins the entries reach the instances PATHS names for them, in both tests:
      k <= 5 canonical {}                MODE_FWD, 8 warps, lane-private replicas (mean length >= 32 kbp in both)
      k <= 5 {"fwd_replicas": 0}         MODE_FWD, 8 warps, no replicas
      k <= 5 {"long_warps": 4}           MODE_FWD, 4 warps
      k = 8 canonical {}                 MODE_K8 with 8 warps, then seq_kernel mode 7 for members over 65535 windows
    seq_kernel, wave_kernel and the multi-launch waves pick their CTA size, grab and tile count from the mean length
    too; those choices change no kernel instance and are left to the heuristics (at 2^32: 256 threads, grab 1, 4096
    tiles per sequence)."""
    p = dict(opts)
    if mins and k <= 5:
        p.setdefault("fwd_min_len", 0)
        p.setdefault("long_warps", 8)
    if mins and k == 8:
        p.setdefault("long_warps", 8)
    return p


# ---------------------------------------------------------------------------------------------------------------------
# base positions past 2^31 and 2^32

P31, P32 = 1 << 31, 1 << 32
_big = None


def big():
    """One 4.06 GiB uint8 buffer of ACGT repeats: bytes next to a batch are valid bases, so counting outside
    [offsets[0], offsets[n]) changes a row."""
    global _big
    if _big is None:
        _big = torch.empty(P32 + (64 << 20), dtype=torch.uint8, device=DEV)
        _big.view(torch.int32).fill_(int.from_bytes(b"ACGT", "little"))
    return _big


def _body(k):
    """Groups of 16 short reads (short_kernel; the groups with a long member go to its reject list), 10 kbp reads
    (MODE_K7 / MODE_K8), 300 kbp contigs (MODE_FWD replicas) and 2 Mbp members (several bucket_kernel tiles), some
    with N runs and IUPAC noise.  Fewer members from k = 9 on, where a row is 0.5 MB or more."""
    rng = np.random.default_rng(4000 + k)
    small_k = k <= 8
    longs = [_seq(rng, 10_000, 0.002, 0.3) for _ in range(8 if small_k else 3)]
    longs += [_seq(rng, 300_000, 0.0005, 0.5) for _ in range(6 if small_k else 2)]
    longs += [_seq(rng, 2_000_000, 0.0002, 0.5) for _ in range(2)]
    rng.shuffle(longs)
    out = []
    for m in longs:
        out += [_seq(rng, int(rng.integers(100, 251)), 0.01, 0.1) for _ in range(31 if small_k else 2)]
        out.append(m)
    return out


def high_batches(k):
    """(members, index of the pinned member, its absolute start) of the three layouts:
      2^31 straddle : a 16 bp member from 2^31 - 7 to 2^31 + 9 between sub-k and empty members
      2^32 exact    : a 10 kbp member ending exactly at 2^32, two empty ones at 2^32, a 10 kbp member starting there
      2^32 straddle : a 16 bp member from 2^32 - 7 to 2^32 + 9 between sub-k and empty members"""
    rng = np.random.default_rng(5000 + k)
    body = _body(k)
    h = len(body) // 2
    sub = lambda: _acgt(rng, k - 1)   # noqa: E731
    empty = lambda: np.zeros(0, np.uint8)   # noqa: E731
    straddle = [sub(), empty(), _acgt(rng, 16), empty(), sub()]
    exact = [_seq(rng, 10_000, 0.001), empty(), empty(), _seq(rng, 10_000, 0.001)]
    return [("2^31 straddle", body[:h] + straddle + body[h:], h + 2, P31 - 7),
            ("2^32 exact", body[:h] + exact + body[h:], h + 3, P32),
            ("2^32 straddle", body[:h] + straddle + body[h:], h + 2, P32 - 7)]


def place(name, members, j, start):
    """Writes the batch into the big buffer so that member j starts at `start`; d_bases is the start of the buffer."""
    bases, offsets = pack(members)
    at = start - int(offsets[j])
    buf = big()
    assert at >= 0 and at + len(bases) + 64 <= buf.numel()
    buf[at:at + len(bases)].copy_(torch.from_numpy(bases))
    b = Batch(name, bases, offsets, buf, at)
    assert b.total == int(b.d_offsets[-1])
    return b


@pytest.mark.parametrize("k,mins,opts,outputs", PATHS, ids=[_id(c) for c in PATHS])
def test_base_positions_past_2_31_and_2_32(k, mins, opts, outputs):
    """Absolute offsets into one 4 GiB buffer: a kernel that keeps a base position in 32 bits reads the wrong bytes."""
    for name, members, j, start in high_batches(k):
        b = place(name, members, j, start)
        for dtype, norm in outputs:
            checked_call(k, b, mins, norm, dtype, f"{name} k{k} mins={mins} {opts} {np.dtype(dtype).name} norm={norm}",
                         opts=pinned(k, mins, opts))
        torch.cuda.synchronize()   # the next layout overwrites these bytes


# ---------------------------------------------------------------------------------------------------------------------
# every element written, nothing outside

def edge_members(k):
    """Lengths where kernels switch: empty, sub-k, one window, chunk and step boundaries, the short-read limit
    254 + k and one past it, a 1.5 Mbp homopolymer (one bin holds every window; it also lifts the mean length over 32 kbp
    so that the replica variant of MODE_FWD applies) and reads with N runs.  The first 16 members are all short, so
    short_kernel writes empty and sub-k rows as well as the later kernels."""
    rng = np.random.default_rng(6000 + k)
    reads = [_seq(rng, int(rng.integers(100, 251)), 0.01) for _ in range(12)]
    lens = [0, 1, k - 1, k, 15, 16, 17, 254 + k]
    out = [_acgt(rng, n) for n in lens] + reads[:8]
    out += [_acgt(rng, 255 + k), np.zeros(0, np.uint8), _acgt(rng, 511), _acgt(rng, 512), _acgt(rng, 513)]
    out += [_seq(rng, 4096, 0.002), _acgt(rng, k - 1), _seq(rng, 70_001, 0.001, 1.0), reads[8],
            np.full(1_500_000, ord("G"), np.uint8)]
    out += [_seq(rng, 3000, 0.01, 1.0) for _ in range(3)] + reads[9:] + [_acgt(rng, k)]
    return out


_edge = {}


def edge_batch(k, at):
    if (k, at) not in _edge:
        if any(kk != k for kk, _ in _edge):
            _edge.clear()
        _edge[(k, at)] = resident("edge", edge_members(k), at)   # same bytes at both offsets: one oracle
        b = _edge[(k, at)]
        assert b.total // b.n >= 32768
    return _edge[(k, at)]


@pytest.mark.parametrize("at", [0, 4093])
@pytest.mark.parametrize("k,mins,opts,outputs", PATHS, ids=[_id(c) for c in PATHS])
def test_every_element_written_nothing_outside(k, mins, opts, outputs, at):
    """Sentinel rows and totals must be fully overwritten and the guards around them untouched, with d_totals set and
    NULL.  at = 4093: d_bases is 16-byte aligned but the first sequence starts 13 bytes into a chunk."""
    b = edge_batch(k, at)
    for dtype, norm in outputs:
        for totals in (False, True):
            checked_call(k, b, mins, norm, dtype, f"edge@{at} k{k} mins={mins} {opts} {np.dtype(dtype).name} "
                         f"norm={norm} totals={totals}", totals=totals, opts=pinned(k, mins, opts))


# ---------------------------------------------------------------------------------------------------------------------
# several calls in flight on one handle

def small_members(k, seed):
    rng = np.random.default_rng(seed)
    out = [_seq(rng, int(rng.integers(100, 251)), 0.01, 0.1) for _ in range(32)]
    out += [np.zeros(0, np.uint8), _acgt(rng, k - 1)] + [_seq(rng, 2000, 0.002, 0.5) for _ in range(4)]
    out.insert(20, _seq(rng, 20_000, 0.001, 0.5))
    return out


def large_members(k, seed):
    """Large enough to grow every scratch buffer k uses: the reject list (many groups), the order list of long contigs
    (k = 5: more 40 kbp contigs than CTAs), the overflow list of packed 16-bit counters (k = 8: members over 65535
    windows), the tile / pool / run buffers of the bucket path (2 Mbp members), and wave rows (k >= 9: over 256 rows
    at k = 10, so four bucket waves become two)."""
    rng = np.random.default_rng(seed)
    reads = lambda m: [_seq(rng, int(rng.integers(100, 251)), 0.01, 0.1) for _ in range(m)]   # noqa: E731
    if k == 5:
        out = [_seq(rng, 36_000, 0.0005, 0.2) for _ in range(1300)] + reads(64)
    elif k == 8:
        out = reads(1200) + [_seq(rng, 10_000, 0.002, 0.2) for _ in range(280)] + [_seq(rng, 100_000, 0.001)] * 2
    else:
        out = reads(200 if k == 10 else 150) + [_seq(rng, 10_000, 0.002, 0.2) for _ in range(60 if k == 10 else 46)]
        out += [_seq(rng, 2_000_000, 0.0002, 0.5) for _ in range(4)]
    rng.shuffle(out)
    return out


# small -> large (scratch grows) -> small (stale scratch behind) -> canonical <-> raw -> u32 -> f32 -> f64 -> NORM_PY
SCRIPT = [("small", True, NORM_CLI, np.float32), ("large", True, NORM_CLI, np.float32),
          ("small", True, NORM_CLI, np.float32), ("small", False, NORM_CLI, np.float32),
          ("small", True, NORM_COUNTS, np.uint32), ("large", True, NORM_COUNTS, np.uint32),
          ("small", False, NORM_COUNTS, np.uint32), ("large", True, NORM_CLI, np.float64),
          ("small", True, NORM_CLI, np.float64),
          ("small", False, NORM_PY, np.float64), ("large", True, NORM_PY, np.float32),
          ("small", True, NORM_COUNTS, np.uint32)]
SHORT_SCRIPT = [("large", True, NORM_CLI, np.float32), ("small", True, NORM_CLI, np.float32),
                ("small", False, NORM_COUNTS, np.uint32)]

BACK_TO_BACK = [
    (5, {}),                                        # short_kernel, seq_kernel mode 1, MODE_FWD replicas + order list
    (8, {}),                                        # short_kernel, MODE_K8 + mode 7 overflow, bucket path (raw)
    (9, {"bucket": 0, "wave_persistent": 0}),       # multi-launch waves on the two aux streams, finalize_kernel
    (10, {}),                                       # bucket_kernel + count_kernel on the caller's stream
    (10, {"bucket_waves": 4}),                      # bucket path in waves on the aux streams (two waves of the large batch)
]


def _script(oc, k, batches, script, stream, opts):
    """Enqueues the whole script without a host sync; the fences and batches stay alive until the caller syncs."""
    return [(f"call {i} {name} mins={mins} norm={norm} {np.dtype(dtype).name}", batches[name], mins, norm,
             enqueue(oc, batches[name], mins, norm, dtype, stream=stream, totals=i % 4 != 3, opts=opts))
            for i, (name, mins, norm, dtype) in enumerate(script)]


def _check_all(k, calls):
    for what, b, mins, norm, fence in calls:
        fence.check(*oracle(b, k, mins, norm), what)


@pytest.mark.parametrize("k,opts", BACK_TO_BACK, ids=[f"k{k}-" + ("-".join(f"{a}={v}" for a, v in o.items()) or "default")
                                                      for k, o in BACK_TO_BACK])
def test_back_to_back_calls_on_one_handle(k, opts):
    """Twelve calls on one handle with no host sync between them, on a torch side stream, then a short script on the
    legacy default stream.  Guards against state carried between calls: work counters not reset, scratch freed or
    reused while a queued call still needs it, stale reject / tile / run entries of a larger batch, helper streams not
    joined back into the caller's stream."""
    oc = handle(k, ("b2b", tuple(opts.items())))
    batches = {"small": resident(f"small{k}", small_members(k, 7000 + k)),
               "large": resident(f"large{k}", large_members(k, 7100 + k))}
    side = torch.cuda.Stream(device=DEV)
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):   # the fences are allocated on the stream that uses them
        calls = _script(oc, k, batches, SCRIPT, side, opts)
    side.synchronize()
    _check_all(k, calls)
    del calls
    calls = _script(oc, k, batches, SHORT_SCRIPT, None, opts)
    torch.cuda.synchronize()
    _check_all(k, calls)


# ---------------------------------------------------------------------------------------------------------------------
# several handles at once

def _concurrent(jobs, rounds):
    """jobs: (k, tag, batch, mins, norm, dtype, opts); job j runs on stream j, the jobs' calls alternate."""
    streams = [torch.cuda.Stream(device=DEV) for _ in jobs]
    for s in streams:
        s.wait_stream(torch.cuda.current_stream())
    calls = []
    for r in range(rounds):
        for (k, tag, b, mins, norm, dtype, opts), s in zip(jobs, streams):
            with torch.cuda.stream(s):
                f = enqueue(handle(k, tag), b, mins, norm, dtype, stream=s, opts=opts)
            calls.append((k, f"round {r} k{k} handle {tag} {b.name}", b, mins, norm, f))
    torch.cuda.synchronize()
    for k, what, b, mins, norm, f in sorted(calls, key=lambda c: c[0]):   # the oracle cache holds one k
        f.check(*oracle(b, k, mins, norm), what)


def _reads_and_contigs(k, seed, n10k, extra):
    rng = np.random.default_rng(seed)
    out = [_seq(rng, 10_000, 0.002, 0.3) for _ in range(n10k)] + [_seq(rng, int(rng.integers(100, 251)), 0.01)
                                                                  for _ in range(48)]
    out += [_seq(rng, extra, 0.0005, 0.5), np.zeros(0, np.uint8), _acgt(rng, k - 1)]
    rng.shuffle(out)
    return out


@pytest.mark.parametrize("k", [7, 10])
def test_two_handles_same_k_two_streams(k):
    """k = 7: long_kernel MODE_K7; k = 10: bucket_kernel + count_kernel.  Different batches, calls alternating."""
    a = resident(f"conc{k}a", _reads_and_contigs(k, 8000 + k, 200 if k == 7 else 40, 1_000_000))
    b = resident(f"conc{k}b", _reads_and_contigs(k, 8100 + k, 150 if k == 7 else 30, 600_000))
    _concurrent([(k, "c0", a, True, NORM_CLI, np.float32, {}), (k, "c1", b, True, NORM_COUNTS, np.uint32, {})], rounds=3)


def test_two_handles_different_k_two_streams():
    """k = 5 (short_kernel + long_kernel MODE_FWD) beside k = 9 (bucket path) on one device."""
    a = resident("conc5", _reads_and_contigs(5, 8205, 100, 1_000_000))
    b = resident("conc9", _reads_and_contigs(9, 8209, 30, 600_000))
    _concurrent([(5, "d0", a, True, NORM_CLI, np.float32, {}), (9, "d1", b, True, NORM_CLI, np.float32, {})], rounds=3)


# ---------------------------------------------------------------------------------------------------------------------
# the tensor surface on a sub-batch view

@pytest.mark.parametrize("k", [4, 7, 10])
def test_tensor_surface_on_sub_batch_views(k):
    """vectorise_tensors(bases, offsets[lo:hi + 1]) reads sequences lo..hi-1 of the resident batch in place; its rows
    must be rows lo..hi-1 of the whole call."""
    rng = np.random.default_rng(9000 + k)
    members = [_seq(rng, int(rng.integers(100, 251)), 0.01, 0.1) for _ in range(40 if k < 10 else 16)]
    members += [_seq(rng, n, 0.002, 0.5) for n in (10_000, 70_001, 300_000, 0, k - 1, 4096)]
    rng.shuffle(members)
    b = resident(f"view{k}", members)
    oc = handle(k, "view")
    want, wtot = oracle(b, k, True, NORM_CLI)
    full = oc.vectorise_tensors(b.buf, b.d_offsets, norm_mode=NORM_CLI, mins=True, dtype=torch.float32)
    torch.cuda.synchronize()
    assert_rows_equal(full.cpu().numpy(), want, np.float32, f"k{k} whole batch")
    n = b.n
    for lo, hi in ((0, n), (1, n - 1), (n // 3, 2 * n // 3), (n - 1, n), (5, 5)):
        tot = torch.full((hi - lo,), -1, dtype=torch.int64, device=DEV)
        part = oc.vectorise_tensors(b.buf, b.d_offsets[lo:hi + 1], norm_mode=NORM_CLI, mins=True, dtype=torch.float32,
                                    totals=tot)
        torch.cuda.synchronize()
        assert tuple(part.shape) == (hi - lo, oc.dim(True))
        assert torch.equal(part, full[lo:hi]), f"k{k} rows [{lo}, {hi}) differ from the whole call"
        assert_rows_equal(part.cpu().numpy(), want[lo:hi], np.float32, f"k{k} rows [{lo}, {hi})")
        assert np.array_equal(tot.cpu().numpy().astype(np.uint64), wtot[lo:hi]), f"k{k} totals [{lo}, {hi})"
