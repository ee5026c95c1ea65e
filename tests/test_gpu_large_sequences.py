"""Sequences long enough to leave the fast write-out of every kernel family.  Needs a B200: -m gpu.

Every kernel that writes a row picks one of two instances of its write-out from the divisor of the row: below 2^23
counts become floats through the 2^23 magic constant and the f32 quotient comes from quot_f32; from 2^23 up (2^24 in
finalize_kernel) counts are converted with I2F and divided in f64.  Any chromosome longer than about 8.4 Mbp takes the
second instance.  One batch per k puts members exactly on both sides of each threshold and is run through every kernel
instance the options can select, bit for bit against the f64 oracle.  The host entry point's 2^30-base chunk cap is
crossed at the end of the file."""
import numpy as np
import pytest

from oracle import oracle as O
from tests.test_gpu_parity import OPTION_DEFAULTS, comp
from tests.util import ALPHA, assert_rows_equal, random_batch

pytestmark = pytest.mark.gpu

from kmertools_b200._lib import NORM_CLI, NORM_COUNTS, NORM_PY  # noqa: E402

P22, P23, P24 = 1 << 22, 1 << 23, 1 << 24


def _acgt(rng, n):
    return ALPHA[rng.integers(0, 4, size=n, dtype=np.uint8)]


def _members(k):
    """(name, bases, intended total or None) of the batch of k.  Lengths depend on k so that the valid-window totals
    land on the thresholds; the short members are interleaved with the long ones."""
    rng = np.random.default_rng(1000 + k)
    n_windows = lambda total: total + k - 1   # noqa: E731  length of a sequence of ACGT with `total` windows
    big = [
        ("A 2^23-1", _acgt(rng, n_windows(P23 - 1)), P23 - 1),            # largest divisor of the fast write-out
        ("B 2^23", _acgt(rng, n_windows(P23)), P23),                      # smallest divisor of the f64 write-out
        # one bin holds every window: an odd count above 2^24, which f32 rounds to the even 2^24 ...
        ("C A*(2^24+1)", np.full(n_windows(P24 + 1), ord("A"), np.uint8), P24 + 1),
    ]
    if k >= 11:   # a row is 8 MB or more: the three members that decide the write-out instance
        return big
    big += [
        # ... and one that f32 rounds up (2^24 + 3 -> 2^24 + 4), which rounding toward zero would not
        ("C' C*(2^24+3)", np.full(n_windows(P24 + 3), ord("C"), np.uint8), P24 + 3),
        # four phases: every pair of reverse-complement bins sums to just over 2^23 (2^23 + 2 at k = 4), and for even k
        # two palindromic bins (the zero word of MODE_FWD's fold) hold 2^22 each
        ("D ACGT*(2^22+2)", np.frombuffer(b"ACGT" * (P22 + 2), np.uint8), P24 + 8 - k + 1),
        # IUPAC codes, lower case, raw 0..3 codes and an N run: a total that is not chosen
        ("E noisy 14 Mbp", random_batch(rng, [14_000_000], noise=0.002, n_runs=1.0)[0], None),
        ("G 2^24-1", _acgt(rng, n_windows(P24 - 1)), P24 - 1),            # largest fast divisor of finalize_kernel
        ("H 2^24+1", _acgt(rng, n_windows(P24 + 1)), P24 + 1),            # first divisor f32 cannot hold
        # raw rows of NORM_PY divide by 2 * total: 2^23 - 2, 2^23, 2^23 + 2
        ("P 2^22-1", _acgt(rng, n_windows(P22 - 1)), P22 - 1),
        ("P 2^22", _acgt(rng, n_windows(P22)), P22),
        ("P 2^22+1", _acgt(rng, n_windows(P22 + 1)), P22 + 1),
    ]
    small = [(f"len {n}", _acgt(rng, n), max(0, n - k + 1)) for n in (0, k - 1, k)]
    small += [(f"read {i}", random_batch(rng, [int(rng.integers(100, 251))], noise=0.01)[0], None)
              for i in range(int(rng.integers(20, 41)))]
    out = []
    for i, m in enumerate(big):   # the short kernel and its reject list run alongside the long members
        out.append(m)
        out += small[i::len(big)]
    return out


_batch = {}
_oracle = {}


def batch(k):
    """(bases, offsets, names, intended totals) of k; one k is cached at a time to bound host memory."""
    if k not in _batch:
        _batch.clear()
        _oracle.clear()
        ms = _members(k)
        lengths = [len(b) for _, b, _ in ms]
        offsets = np.zeros(len(ms) + 1, dtype=np.uint64)
        np.cumsum(lengths, out=offsets[1:])
        bases = np.concatenate([b for _, b, _ in ms])
        _batch[k] = (bases, offsets, [m[0] for m in ms], [m[2] for m in ms])
    return _batch[k]


def oracle(k, mins, norm_mode):
    """f64 oracle rows and totals, computed once per (k, mins, norm_mode).  The totals must be the intended ones, so
    that an edit of the generator cannot move a member off its threshold unnoticed."""
    key = (k, mins, norm_mode)
    if key not in _oracle:
        bases, offsets, names, intended = batch(k)
        rows, totals = O.vectorise_batch(bases, offsets, k, mins, norm_mode)
        for name, want, got in zip(names, intended, totals):
            assert want is None or int(got) == want, (k, name, int(got), want)
        if k < 11:
            assert int(totals[names.index("E noisy 14 Mbp")]) > P23
        _oracle[key] = (rows, totals)
    return _oracle[key]


def run(k, mins, norm_mode, dtype, what, **opts):
    """One call through the host entry point with `opts` set (the rest at their defaults), against the oracle."""
    assert set(opts) <= {key for key, _ in OPTION_DEFAULTS}, opts
    bases, offsets, _, _ = batch(k)
    oc = comp(k)
    for key, dflt in OPTION_DEFAULTS:
        oc.set_option(key, opts.get(key, dflt))
    try:
        totals = np.zeros(len(offsets) - 1, dtype=np.uint64)
        got = oc.vectorise_packed(bases, offsets, norm_mode=norm_mode, mins=mins, dtype=dtype, totals=totals)
        want, wtot = oracle(k, mins, norm_mode)
        assert np.array_equal(totals, wtot), f"{what}: totals differ"
        assert_rows_equal(got, want, dtype, what)
    finally:
        for key, dflt in OPTION_DEFAULTS:
            oc.set_option(key, dflt)


U32_F32 = ((np.uint32, NORM_COUNTS), (np.float32, NORM_CLI), (np.float32, NORM_COUNTS))
U32_F32_PY = U32_F32 + ((np.float32, NORM_PY),)
F64 = ((np.float64, NORM_CLI), (np.float64, NORM_COUNTS))
F64_PY = F64 + ((np.float64, NORM_PY),)

# (k, canonical, options, outputs): each entry reaches one kernel instance (noted) with the batch of k.  Ordered by k,
# so that each batch and its oracle rows are built once.
PATHS = [
    *[c for k in (3, 4, 5) for c in (
        (k, True, {}, U32_F32),                       # long_kernel MODE_FWD, lane-private replicas
        (k, True, {"fwd_replicas": 0}, U32_F32),      # MODE_FWD without replicas
        (k, True, {"long_warps": 4}, U32_F32),        # MODE_FWD with 4 warps per CTA
        (k, True, {"fwd_fold": 0}, U32_F32),          # seq_kernel mode 1
        (k, True, {}, F64),                           # seq_kernel mode 1 (long_kernel has no f64 instance)
        *([(4, False, {}, U32_F32_PY + F64_PY),       # seq_kernel mode 0
           (4, True, {"force_path": 1}, U32_F32 + F64)] if k == 4 else []),   # flat_kernel + finalize_kernel
    )],
    (6, True, {}, U32_F32 + F64),                     # seq_kernel mode 1
    (6, True, {"fwd_fold": 0}, U32_F32),
    (7, True, {}, U32_F32),                           # long_kernel MODE_K7
    (7, True, {"k7_mid": 0}, U32_F32 + F64),          # seq_kernel mode 4 (also the f64 default)
    (7, True, {"k7_mid": 0, "dense_odd": 0}, U32_F32),   # seq_kernel mode 1
    (7, False, {}, U32_F32_PY + F64_PY),              # seq_kernel mode 0
    (8, True, {}, U32_F32),                           # long_kernel MODE_K8, every long member to seq_kernel mode 7
    (8, True, {"k8_long": 0}, U32_F32 + F64),         # seq_kernel mode 5, then mode 7 (also the f64 default)
    (8, True, {"packed16": 0}, U32_F32),              # seq_kernel mode 7 directly
    (8, True, {"even_rank": 0}, U32_F32),             # seq_kernel mode 2
    (8, False, {}, U32_F32_PY + F64_PY),              # bucket_kernel + count_kernel, raw
    (8, False, {"bucket": 0}, U32_F32_PY),            # wave_kernel RANK 0
    (9, True, {}, U32_F32 + F64),                     # bucket_kernel + count_kernel
    (9, True, {"bucket_log2_seg": 13}, U32_F32),      # count_kernel with two 2^13-bin buffers
    (9, True, {"bucket": 0}, U32_F32),                # wave_kernel RANK 2
    (9, True, {"bucket": 0, "wave_smem_rank": 0}, U32_F32),   # wave_kernel RANK 1
    (9, True, {"bucket": 0, "wave_persistent": 0}, U32_F32),  # seq_kernel mode 3 waves + finalize_kernel
    (9, True, {"bucket": 0}, F64),                    # seq_kernel mode 3 waves + finalize_kernel
    (9, True, {"force_path": 1}, U32_F32 + F64),      # flat_kernel + finalize_kernel
    (9, False, {}, U32_F32_PY + F64_PY),              # bucket_kernel + count_kernel, raw
    (10, True, {}, U32_F32 + F64),                    # bucket_kernel + count_kernel
    (10, True, {"bucket": 0}, U32_F32),               # wave_kernel RANK 2
    (11, True, {}, U32_F32),                          # wave_kernel RANK 1 (members A-C)
]


def _id(c):
    k, mins, opts, _ = c
    return f"k{k}-{'canon' if mins else 'raw'}-" + ("-".join(f"{a}={b}" for a, b in opts.items()) or "default") + \
        ("-f64" if c[3][0][0] is np.float64 else "")


@pytest.mark.parametrize("k,mins,opts,outputs", PATHS, ids=[_id(c) for c in PATHS])
def test_large_divisor_write_out(k, mins, opts, outputs):
    for dtype, norm in outputs:
        run(k, mins, norm, dtype, f"k{k} mins={mins} {opts} {np.dtype(dtype).name} norm={norm}", **opts)


def test_device_entry_point_large_sequences():
    """The torch-owned path (CUDA tensors in and out) on the k = 10 batch."""
    import torch
    bases, offsets, _, _ = batch(10)
    oc = comp(10)
    dev = torch.device("cuda:0")
    tb = torch.from_numpy(bases).to(dev)
    to = torch.from_numpy(offsets.astype(np.int64)).to(dev)
    tot = torch.zeros(len(offsets) - 1, dtype=torch.int64, device=dev)
    out = oc.vectorise_tensors(tb, to, norm_mode=NORM_CLI, mins=True, dtype=torch.float32, totals=tot)
    torch.cuda.synchronize()
    want, wtot = oracle(10, True, NORM_CLI)
    assert_rows_equal(out.cpu().numpy(), want, np.float32, "device path k10")
    assert np.array_equal(tot.cpu().numpy().astype(np.uint64), wtot)


# ---------------------------------------------------------------------------------------------------------------------
# the host entry point copies at most 2^30 bases per chunk

def test_chunk_cap_splits_many_sequences():
    """320 sequences of 3.5 Mbp (1.12 GB): the rows fit one row chunk, so only the base cap splits the batch.  Every
    sequence is random with an N run of its own, so a row written to the wrong place differs."""
    _batch.clear()
    _oracle.clear()
    n, L, k = 320, 3_500_000, 4
    rng = np.random.default_rng(31)
    offsets = np.arange(n + 1, dtype=np.uint64) * np.uint64(L)
    bases = np.empty(n * L, dtype=np.uint8)
    for i in range(n):
        s = bases[i * L:(i + 1) * L]
        s[:] = _acgt(rng, L)
        a = int(rng.integers(0, L - 200_000))
        s[a:a + int(rng.integers(1, 200_000))] = ord("N")
    assert int(offsets[-1]) > 1 << 30 and n * comp(k).dim(True) * 4 < 512 << 20
    for dtype, norm in ((np.uint32, NORM_COUNTS), (np.float32, NORM_CLI)):
        totals = np.zeros(n, dtype=np.uint64)
        got = comp(k).vectorise_packed(bases, offsets, norm_mode=norm, mins=True, dtype=dtype, totals=totals)
        want, wtot = O.vectorise_batch(bases, offsets, k, True, norm)
        assert np.array_equal(totals, wtot), "totals differ"
        assert_rows_equal(got, want, dtype, f"chunk cap {np.dtype(dtype).name}")


def test_chunk_cap_one_sequence_beyond_it():
    """[150 bp, 1.1 Gbp, 150 bp]: the middle chunk holds exactly one sequence larger than the cap."""
    k, L = 4, 1_100_000_000
    rng = np.random.default_rng(32)
    offsets = np.array([0, 150, 150 + L, 300 + L], dtype=np.uint64)
    bases = np.empty(300 + L, dtype=np.uint8)
    step = 1 << 26
    for a in range(0, bases.size, step):
        bases[a:a + step] = _acgt(rng, min(step, bases.size - a))
    bases[150 + L // 3:150 + L // 3 + 5000] = ord("N")
    for dtype, norm in ((np.uint32, NORM_COUNTS), (np.float32, NORM_CLI)):
        totals = np.zeros(3, dtype=np.uint64)
        got = comp(k).vectorise_packed(bases, offsets, norm_mode=norm, mins=True, dtype=dtype, totals=totals)
        want, wtot = O.vectorise_batch(bases, offsets, k, True, norm)
        assert np.array_equal(totals, wtot), "totals differ"
        assert_rows_equal(got, want, dtype, f"one sequence beyond the cap {np.dtype(dtype).name}")
