"""Every launch shape the tuning options reach, and the rows no other test builds.  Needs a B200: -m gpu.

The other parity tests run each kernel instance at the shape its heuristic picks for their batches.  The options of
`ktb_oligo_set_option` reach further: the CTA size and grab of seq_kernel (`seq_threads`, `seq_grab`), the tiling of
the multi-launch wave loop (`global_steps_per_warp`), the warps of long_kernel (`long_warps`), the histogram memory and
the waves of the bucket path (`bucket_hist_kb`, `bucket_log2_seg`, `bucket_waves`, `bucket_wave_ctas`).  Raw rows at
k = 10, 11, 12 and f64 rows at canonical k = 10, 11, 12 are built here too.  Every case compares rows and totals bit
for bit with the f64 oracle, and where the number of launches pins the path it asserts that number, so that a case
cannot pass on the default path.  The expected counts follow the launchers of csrc/api.cu (see `host_launches`)."""
import numpy as np
import pytest

from oracle import oracle as O
from tests.test_gpu_parity import OPTION_DEFAULTS, comp
from tests.util import assert_rows_equal, random_batch

pytestmark = pytest.mark.gpu

from kmertools_b200._lib import NORM_CLI, NORM_COUNTS, NORM_PY  # noqa: E402

# OPTION_DEFAULTS and the four options it leaves out, at their defaults
DEFAULTS = OPTION_DEFAULTS + (("seq_threads", 0), ("seq_grab", 0), ("global_steps_per_warp", 1),
                              ("bucket_wave_ctas", 2))
CHUNK_BYTES = 512 << 20         # default "chunk_bytes": output bytes per chunk of the host entry point
GLOBAL_WAVE_BYTES = 64 << 20    # default "global_wave_bytes"
TILE = 248 * 16                 # bases per tile of bucket_kernel
ORACLE_CACHE_BYTES = 3 << 29   # oracle rows kept for the outputs of one batch and k (a raw k = 12 f64 row is 128 MiB)

U32_F32 = ((np.uint32, NORM_COUNTS), (np.float32, NORM_CLI))
U32_F32_PY = U32_F32 + ((np.float32, NORM_PY),)
F64 = ((np.float64, NORM_CLI), (np.float64, NORM_PY))

_touched = set()


def set_options(oc, opts):
    """Sets every option of DEFAULTS on `oc`: the value in `opts`, else the default."""
    assert set(opts) <= {key for key, _ in DEFAULTS}, opts
    for key, dflt in DEFAULTS:
        oc.set_option(key, opts.get(key, dflt))


@pytest.fixture(scope="module", autouse=True)
def _restore_options():
    """The handles are shared with the other modules: leave every option of every handle used here at its default."""
    yield
    for k in sorted(_touched):
        set_options(comp(k), {})
    _batch.clear()
    _oracle.clear()


# ---------------------------------------------------------------------------------------------------------------------
# launches of one call through the host entry point, per chunk of rows, as the launchers of csrc/api.cu enqueue them

def fixed(count):
    """The shared-memory histogram paths: short_kernel (k <= 5) and the CTA-per-sequence kernels, a fixed number."""
    return lambda cn, dim, dtype: count


def wave_loop(cn, dim, dtype):
    """launch_wave_loop: waves of rows that fill half of "global_wave_bytes" (at least one row); per wave seq_kernel
    mode 3, and finalize_kernel unless the output is u32."""
    wave = max(1, min(cn, GLOBAL_WAVE_BYTES // 2 // (dim * 4)))
    return -(-cn // wave) * (1 if np.dtype(dtype) == np.uint32 else 2)


def bucket(waves):
    """launch_bucket: tile_prefix_kernel + tile_info_kernel, then bucket_kernel + count_kernel per wave; the waves
    are min("bucket_waves", chunks of 8 sequences / 16), at least one."""
    return lambda cn, dim, dtype: 2 + 2 * max(1, min(waves, -(-cn // 8) // 16))


def coop_or_loop(cn, dim, dtype):
    """Rows larger than shared memory outside the bucket path: one cooperative wave_kernel for u32 / f32 rows, the
    wave loop for f64 rows."""
    return wave_loop(cn, dim, dtype) if np.dtype(dtype) == np.float64 else 1


def host_launches(per_chunk, offsets, dim, dtype):
    """ktb_oligo_vectorise cuts the batch into chunks of CHUNK_BYTES of output rows and adds one rebase_offsets_kernel
    for each chunk whose first base is not in the first 16 bytes of the batch."""
    n = len(offsets) - 1
    assert int(offsets[-1]) <= 1 << 30   # no chunk is cut by the 2^30-base cap
    rows = max(1, CHUNK_BYTES // (dim * np.dtype(dtype).itemsize))
    total = 0
    for i0 in range(0, n, rows):
        total += per_chunk(min(rows, n - i0), dim, dtype) + ((int(offsets[i0]) & ~15) != 0)
    return total


# ---------------------------------------------------------------------------------------------------------------------
# batches and oracle rows (one batch, and the rows of one batch and k, are kept at a time)

_batch = {}
_oracle = {}


def batch(name, k):
    if (name, k) not in _batch:
        _batch.clear()
        _oracle.clear()
        _batch[(name, k)] = BATCHES[name](k)
    return _batch[(name, k)]


def oracle(name, k, mins, norm):
    key = (name, k, mins, norm)
    if key not in _oracle:
        bases, offsets = batch(name, k)
        new = (len(offsets) - 1) * O.dim(k, mins) * 8
        if any(kk[:3] != key[:3] for kk in _oracle) or \
                sum(r.nbytes for r, _ in _oracle.values()) + new > ORACLE_CACHE_BYTES:
            _oracle.clear()
        _oracle[key] = O.vectorise_batch(bases, offsets, k, mins, norm)
    return _oracle[key]


def mixed(k):
    """Groups of 16 reads of 150 ... 254 + k bases (the longest read short_kernel takes), every third one with a longer
    member so that short_kernel puts it on the reject list; members of length 0, k - 1 and k; 1 ... 20 kbp members;
    one member of 70,001 bases (more than 65,535 windows at k = 8).  Fewer groups at k = 9, whose rows are 0.5 MB."""
    rng = np.random.default_rng(500 + k)
    lengths = []
    for g in range(24 if k < 9 else 4):
        grp = [int(x) for x in rng.integers(150, 255 + k, size=16)]
        if g % 4 == 0:
            grp[int(rng.integers(0, 16))] = 254 + k
        if g % 3 == 1:
            grp[int(rng.integers(0, 16))] = 255 + k if g == 1 else int(rng.integers(256 + k, 3000))
        lengths += grp
    lengths += [0, k - 1, k, *(int(x) for x in rng.integers(1000, 20_001, size=16)), 70_001]
    return random_batch(rng, lengths, noise=0.003, n_runs=0.2)


def contig(k):
    """17.5 Mbp and a member of k - 1 bases: a mean length of 8.75 Mbp, 17,090 steps of 512 bases."""
    rng = np.random.default_rng(600 + k)
    return random_batch(rng, [17_500_000, k - 1], noise=0.001, n_runs=1.0)


def contigs(k):
    """1,300 contigs of 8 ... 120 kbp (mean above 32 kbp, more contigs than long_kernel has CTAs), every 97th a read
    short enough for short_kernel, one empty."""
    rng = np.random.default_rng(700 + k)
    lengths = np.exp(rng.uniform(np.log(8e3), np.log(1.2e5), size=1300)).astype(np.int64)
    lengths[::97] = rng.integers(0, 200, size=len(lengths[::97]))
    lengths[5] = 0
    return random_batch(rng, lengths, noise=0.002, n_runs=0.5)


def ragged(k):
    """Lengths around 16-byte chunks and bucket_kernel tiles, a 120 kbp member and a homopolymer (one segment run, one
    bin)."""
    rng = np.random.default_rng(800 + k)
    lengths = np.r_[rng.integers(0, 4000, size=24), [0, 1, k - 1, k, 15, 16, 17, TILE - 1, TILE, TILE + 1,
                                                      3 * TILE + 500, 120_000, 20_000]]
    bases, offsets = random_batch(rng, lengths, noise=0.003, n_runs=0.2)
    bases[int(offsets[-2]):] = ord("A")
    return bases, offsets


def many(k):
    """700 reads of 100 ... 3000 bases: 88 chunks of 8 sequences, enough for five waves of the bucket path."""
    rng = np.random.default_rng(900 + k)
    lengths = np.r_[rng.integers(100, 3000, size=697), [0, k - 1, k]]
    rng.shuffle(lengths)
    return random_batch(rng, lengths, noise=0.003, n_runs=0.1)


def few(k):
    """Eight members: 0, k - 1 and k bases, 700, 5000 and 200,000 bases of noisy ACGT, 3,000 bases with an N run of
    1,000 in the middle, and a 20,000-base homopolymer."""
    rng = np.random.default_rng(1000 + k)
    bases, offsets = random_batch(rng, [0, k - 1, k, 700, 5000, 200_000, 3000, 20_000], noise=0.002)
    bases[int(offsets[6]) + 1000:int(offsets[6]) + 2000] = ord("N")
    bases[int(offsets[7]):] = ord("C")
    return bases, offsets


BATCHES = {"mixed": mixed, "contig": contig, "contigs": contigs, "ragged": ragged, "many": many, "few": few}


def run(name, k, mins, opts, outputs, per_chunk):
    """Each output of the batch `name` through the host entry point with `opts` set (every other option at its
    default), against the oracle; the launches of the call against `per_chunk`."""
    bases, offsets = batch(name, k)
    n = len(offsets) - 1
    oc = comp(k)
    _touched.add(k)
    for dtype, norm in outputs:
        what = f"{name} k{k} {'canon' if mins else 'raw'} {opts} {np.dtype(dtype).name} norm={norm}"
        totals = np.zeros(n, dtype=np.uint64)
        set_options(oc, opts)
        try:
            got = oc.vectorise_packed(bases, offsets, norm_mode=norm, mins=mins, dtype=dtype, totals=totals)
            launches = oc.stats()["launches"]
        finally:
            set_options(oc, {})
        want, wtot = oracle(name, k, mins, norm)
        assert np.array_equal(totals, wtot), f"{what}: totals differ"
        assert_rows_equal(got, want, dtype, what)
        del got
        expected = host_launches(per_chunk, offsets, oc.dim(mins), dtype)
        assert launches == expected, f"{what}: {launches} launches, expected {expected}"


def case_id(instance, k, mins, opts, outputs):
    return f"{instance}-k{k}-{'canon' if mins else 'raw'}-" + \
        ("-".join(f"{a}={b}" for a, b in opts.items()) or "default") + \
        ("-f64" if all(np.dtype(d) == np.float64 for d, _ in outputs) else "")


# ---------------------------------------------------------------------------------------------------------------------
# a. seq_kernel: CTA size and grab, in every mode

# (instance, k, canonical, options, outputs, launches per chunk)
SEQ_MODES = [
    ("seq_kernel-mode0", 4, False, {"force_path": 2}, U32_F32_PY, fixed(1)),
    ("short_kernel+seq_kernel-mode1", 4, True, {"fwd_fold": 0}, U32_F32_PY, fixed(2)),   # f32 norm: KT = 4
    ("short_kernel+seq_kernel-mode1", 5, True, {"fwd_fold": 0}, U32_F32_PY, fixed(2)),   # f32 norm: KT = 5
    ("seq_kernel-mode1", 6, True, {}, U32_F32_PY, fixed(1)),                              # f32 norm: KT = 6
    ("seq_kernel-mode0", 7, False, {}, U32_F32_PY, fixed(1)),
    ("seq_kernel-mode4", 7, True, {"k7_mid": 0}, U32_F32_PY, fixed(1)),                  # f32 norm: KT = 7
    ("seq_kernel-mode5+mode7", 8, True, {"k8_long": 0}, U32_F32_PY, fixed(2)),
    ("seq_kernel-mode7", 8, True, {"packed16": 0}, U32_F32_PY, fixed(1)),
    ("seq_kernel-mode2", 8, True, {"even_rank": 0}, U32_F32_PY, fixed(1)),
    ("seq_kernel-mode3-waves", 9, True, {"bucket": 0, "wave_persistent": 0}, U32_F32_PY, wave_loop),
    ("seq_kernel-mode3-waves", 9, True, {"bucket": 0}, F64, wave_loop),
]
# 96 is no power of two; 512 and 1024 are above the launch bound of modes 0, 1, 3, 4 and 5, which clamp them.  The
# wave loop (mode 3) takes one item per trip to the work counter whatever "seq_grab" says.
SEQ_SHAPES = [*({"seq_threads": t} for t in (32, 96, 256, 512, 1024)), *({"seq_grab": g} for g in (1, 7, 1024)),
              {"seq_threads": 96, "seq_grab": 7}]
SEQ_CASES = [(inst, k, mins, {**opts, **shape}, outs, per)
             for inst, k, mins, opts, outs, per in SEQ_MODES for shape in SEQ_SHAPES]


@pytest.mark.parametrize("instance,k,mins,opts,outputs,per_chunk", SEQ_CASES,
                         ids=[case_id(*c[:5]) for c in SEQ_CASES])
def test_seq_kernel_cta_size_and_grab(instance, k, mins, opts, outputs, per_chunk):
    run("mixed", k, mins, opts, outputs, per_chunk)


# ---------------------------------------------------------------------------------------------------------------------
# b. the wave loop's tiles: about "global_steps_per_warp" steps of 512 bases per warp, at most 4096 tiles a sequence

WAVE_LOOP = [("seq_kernel-mode3-waves", 9, True, {"bucket": 0, "wave_persistent": 0}, U32_F32_PY),
             ("seq_kernel-mode3-waves", 9, True, {"bucket": 0}, F64)]
TILE_CASES = [(name, inst, k, mins, {**opts, "global_steps_per_warp": g}, outs)
              for name in ("mixed", "contig") for inst, k, mins, opts, outs in WAVE_LOOP for g in (1, 3, 64)]


@pytest.mark.parametrize("name,instance,k,mins,opts,outputs", TILE_CASES,
                         ids=[f"{c[0]}-" + case_id(*c[1:]) for c in TILE_CASES])
def test_wave_loop_tiles(name, instance, k, mins, opts, outputs):
    if name == "contig" and opts["global_steps_per_warp"] == 1:
        bases, offsets = batch(name, k)
        mean_steps = int(offsets[-1]) // (len(offsets) - 1) // 512 + 1
        assert mean_steps // (128 // 32) > 4096   # 128 threads, one step per warp: the tile count is capped
    run(name, k, mins, opts, outputs, wave_loop)


# ---------------------------------------------------------------------------------------------------------------------
# c. long_kernel: 4, 8 and 10 warps; 10 is 8 outside MODE_K7, and the replica variant needs 8

LONG_CASES = [
    *(("mixed", f"long_kernel-K7-w{w}", 7, {"long_warps": w}, fixed(1)) for w in (4, 8, 10)),
    *(("mixed", "short_kernel+long_kernel-FWD-w8", k, {"fwd_min_len": 0, "long_warps": 10}, fixed(2))
      for k in (3, 4, 5)),
    ("mixed", "long_kernel-K8-w8+seq_kernel-mode7", 8, {"long_warps": 10}, fixed(2)),
    # mean length >= 32 kbp: with 4 warps the plain MODE_FWD kernel, input order; with 10 (= 8) the replicas, and
    # more contigs than CTAs hand the long ones out first (order_count_kernel + order_scatter_kernel)
    *(c for k in (3, 4, 5) for c in (
        ("contigs", "short_kernel+long_kernel-FWD-w4", k, {"long_warps": 4}, fixed(2)),
        ("contigs", "short_kernel+order+long_kernel-FWD-w8-replicas", k, {"long_warps": 10}, fixed(4)))),
]


@pytest.mark.parametrize("name,instance,k,opts,per_chunk", LONG_CASES,
                         ids=[f"{c[0]}-" + case_id(c[1], c[2], True, c[3], U32_F32_PY) for c in LONG_CASES])
def test_long_kernel_warps(name, instance, k, opts, per_chunk):
    if name == "contigs":
        import torch
        bases, offsets = batch(name, k)
        n = len(offsets) - 1
        assert bases.size // n >= 32768
        assert n > torch.cuda.get_device_properties(0).multi_processor_count * 8   # 8 CTAs of 256 threads fill an SM
    run(name, k, True, opts, U32_F32_PY, per_chunk)


# ---------------------------------------------------------------------------------------------------------------------
# d. the bucket path: 96 KB of count_kernel histogram, both segment sizes, 128 segments, waves

BUCKET_CASES = [
    *(("ragged", "bucket+count_kernel-hist96", k, mins, {"bucket_hist_kb": 96, "bucket_log2_seg": s}, U32_F32_PY, 1)
      for k, mins in ((9, True), (10, True), (8, False), (9, False), (10, False)) for s in (13, 14)),
    # canonical k = 9 in segments of 2^14 codes: 4 of 16 segments hold more than 12,288 columns
    ("ragged", "bucket+count_kernel-hist96", 9, True, {"bucket_hist_kb": 96, "bucket_log2_seg": 14}, F64, 1),
    # raw k = 10 in segments of 2^13 codes: 128 segments, BK_MAX_SEG
    ("ragged", "bucket+count_kernel-128seg", 10, False, {"bucket_log2_seg": 13}, U32_F32_PY + F64, 1),
    *(("many", f"bucket+count_kernel-{w}waves", 8, False, {"bucket_waves": w, "bucket_wave_ctas": c},
       U32_F32_PY + (F64 if (w, c) == (5, 4) else ()), w) for w in (2, 5) for c in (1, 4)),
]


@pytest.mark.parametrize("name,instance,k,mins,opts,outputs,waves", BUCKET_CASES,
                         ids=[f"{c[0]}-" + case_id(*c[1:6]) + ("-with-f64" if len(c[5]) > 3 else "")
                              for c in BUCKET_CASES])
def test_bucket_path_shapes(name, instance, k, mins, opts, outputs, waves):
    run(name, k, mins, opts, outputs, bucket(waves))


# ---------------------------------------------------------------------------------------------------------------------
# e. rows that no other test builds, default options

ROW_CASES = [
    ("bucket+count_kernel", 10, False, U32_F32_PY + F64, bucket(1)),
    ("wave_kernel-RANK0+f64:seq_kernel-mode3", 11, False, U32_F32 + F64, coop_or_loop),
    ("wave_kernel-RANK0+f64:seq_kernel-mode3", 12, False, U32_F32 + F64, coop_or_loop),
    ("bucket+count_kernel", 10, True, F64, bucket(1)),
    ("seq_kernel-mode3-waves", 11, True, F64, wave_loop),
    ("wave_kernel-RANK1+f64:seq_kernel-mode3", 12, True, ((np.float32, NORM_PY),) + F64, coop_or_loop),
]


@pytest.mark.parametrize("instance,k,mins,outputs,per_chunk", ROW_CASES,
                         ids=[case_id(c[0], c[1], c[2], {}, c[3]) for c in ROW_CASES])
def test_rows_of_large_k(instance, k, mins, outputs, per_chunk):
    """A raw k = 12 f64 row is 128 MiB: the host entry point takes four rows per chunk, and the oracle keeps the rows
    of one output at a time."""
    run("few", k, mins, {}, outputs, per_chunk)
