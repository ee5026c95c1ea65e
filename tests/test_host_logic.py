"""CPU-side checks of host logic and of arithmetic claims the kernels rely on."""
import numpy as np
import pytest

from oracle import oracle as O


def test_f32_division_sequence_is_correctly_rounded():
    """DESIGN.md §5: q0 = c*RN(1/d); q = fma(fma(-q0,d,c), RN(1/d), q0) == (float)((double)c/(double)d).
    Exhaustive for every divisor a short read (<= 510) or a 4 kbp sequence can produce, sampled above."""
    assert O.check_quot_f32(1, 4096, 1) == 0
    assert O.check_quot_f32(4097, 70000, 997) == 0
    assert O.check_quot_f32((1 << 24) - 300, (1 << 24) - 1, 65537) == 0


def test_bench_algorithmic_bytes_formula():
    import bench
    # SURVEY §8(d): config 2 = 22.06 GB, config 3 = 42.78 GB
    assert bench.algorithmic_bytes(1_500_000_000, 10_000_000, 512, 4) == 22_060_000_008
    assert abs(bench.algorithmic_bytes(10_000_000_000, 1_000_000, 8192, 4) - 42.78e9) < 0.01e9
    assert [bench.dim_of(k) for k in (3, 4, 5, 6, 7, 8, 10)] == [32, 136, 512, 2080, 8192, 32896, 524800]


def test_bench_dump_rows_is_a_fixed_sample_within_the_cap(tmp_path):
    """--dump-outputs: small outputs are written whole; large ones as the same seeded row sample every run, under
    DUMP_BYTES; f32 rows stay float32, u32 counts become exact float64."""
    import torch
    import bench
    small = torch.arange(6 * 32, dtype=torch.int32).view(6, 32)
    bench.dump_rows(small, "u32", tmp_path / "s.npy")
    got = np.load(tmp_path / "s.npy")
    assert got.dtype == np.float64 and np.array_equal(got, small.numpy())
    big = torch.rand(2 * bench.DUMP_BYTES // (512 * 4), 512, generator=torch.Generator().manual_seed(0))
    bench.dump_rows(big, "f32", tmp_path / "a.npy")
    bench.dump_rows(big, "f32", tmp_path / "b.npy")
    a, b = np.load(tmp_path / "a.npy"), np.load(tmp_path / "b.npy")
    assert a.dtype == np.float32 and a.shape == (bench.DUMP_BYTES // (512 * 4), 512) and np.array_equal(a, b)
    assert (tmp_path / "a.npy").stat().st_size <= bench.DUMP_BYTES + 4096
    pick = np.sort(np.random.default_rng(bench.DUMP_SEED).choice(len(big), size=len(a), replace=False))
    assert np.array_equal(a, big.numpy()[pick]) and len(np.unique(pick)) == len(a)


def test_pack_helper_matches_oracle_pack():
    from kmertools_b200.oligo import _pack
    seqs = ["ACGT", "", "NNACGTTT", "acgu"]
    b1, o1 = _pack(seqs)
    b2, o2 = O.pack([s.encode() for s in seqs])
    assert np.array_equal(b1, b2) and np.array_equal(o1, o2)


def test_shard_bounds_matches_the_python_sharder():
    """ktb_shard_bounds (the product's partition, csrc/multi.cu) == kmertools_b200.shard.shard_by_bases: contiguous,
    complete, monotone, balanced by bases; by count when every sequence is empty."""
    from kmertools_b200 import shard_bounds
    from kmertools_b200.shard import shard_by_bases
    from tests.util import random_batch
    rng = np.random.default_rng(5)
    cases = [rng.integers(0, 400, size=300), np.r_[rng.integers(0, 50, size=40), [90_000], rng.integers(0, 50, size=40)],
             np.zeros(17, dtype=np.int64), np.array([5]), np.array([], dtype=np.int64), np.full(1000, 150)]
    for lengths in cases:
        _, offsets = random_batch(rng, lengths)
        for shift in (0, 37):
            offs = offsets + np.uint64(shift)
            for parts in (1, 2, 3, 8):
                b = shard_bounds(offs, parts)
                assert b[0] == 0 and b[-1] == len(lengths) and np.all(np.diff(b.astype(np.int64)) >= 0)
                for r in range(parts):
                    assert (int(b[r]), int(b[r + 1])) == shard_by_bases(offs, parts, r)
                if len(lengths) and lengths.sum():
                    per = [int(offs[b[r + 1]]) - int(offs[b[r]]) for r in range(parts)]
                    assert max(per) - lengths.sum() / parts <= lengths.max()


def test_bench_generator_is_backend_independent_and_prefix_stable():
    """bench.py's workloads are hashes of (seed, position / read index): numpy and torch produce the same bytes, and
    the first m sequences do not depend on how many follow — so the CPU arms time a prefix of the GPU arm's data."""
    import torch
    import bench
    for name, scale in (("reads150_k5", 0.0005), ("reads10k_k7", 0.0003), ("contigs_k4", 0.004), ("reads100k_k10", 0.02)):
        spec = bench.WORKLOADS[name]
        bn, on = bench.make_workload(spec, scale, bench._NP())
        bt, ot = bench.make_workload_torch(spec, scale, torch.device("cpu"))
        assert np.array_equal(bn, bt.numpy()) and np.array_equal(on, ot.numpy()), name
        m = 7
        bp, op = bench.make_workload(spec, scale, bench._NP(), n_limit=m)
        assert np.array_equal(op, on[: m + 1]) and np.array_equal(bp, bn[: int(on[m])]), name
        cfg = bench.config_of(name, spec, scale)
        assert cfg["sequences_per_gpu"] == len(on) - 1 and cfg["bases_per_gpu"] == int(on[-1])
        # the alphabet the config promises
        letters = set(bytes(bn.tobytes()))
        assert letters >= set(b"ACGT") and ord("N") in letters or name == "reads100k_k10"
    spec = bench.WORKLOADS["contigs_k4"]
    b, o = bench.make_workload(spec, 0.01, bench._NP())
    L = np.diff(o)
    assert L.min() >= 1000 and L.max() <= 500_000
    frac_n = float((b == ord("N")).mean())
    assert 0.0 < frac_n < 0.2 and (np.isin(b, list(b"acgt"))).mean() > 0.01 and np.isin(b, list(b"RYKMSW")).any()
