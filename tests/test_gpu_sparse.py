"""Sparse (CSR) k-mer count rows on the GPU, bit for bit: against the dense rows and the oracle for k <= 12, against the
oracle restatement (tests/sparse_ref.py) up to k = 31, at tile and merge boundaries, and through the device entry point
(sub-batch views, offsets past 2^32, fenced outputs, cap, two streams, determinism)."""

import numpy as np
import pytest

from kmertools_b200 import OligoComputer, _lib, kmer_counts, kmer_counts_tensors
from oracle import oracle
from tests.sparse_ref import scatter, sparse_rows
from tests.util import random_batch

pytestmark = pytest.mark.gpu

T = 4096   # positions per tile of sparse_tile_kernel
DT = {0: np.uint32, 1: np.float32, 2: np.float64}
COMBOS = [(0, 0), (0, 1), (1, 1), (2, 1), (0, 2), (1, 2), (2, 2)]   # (norm_mode, out_dtype)


def check_against_ref(bases, offsets, k, canonical, norm, dtype, got=None, what=""):
    rp, codes, vals, tot = got if got is not None else kmer_counts((bases, offsets), k, canonical, norm, dtype)
    w_rp, w_codes, w_vals, w_tot = sparse_rows(bases, offsets, k, canonical, norm)
    assert np.array_equal(tot, w_tot), what
    assert np.array_equal(rp, w_rp), what
    assert np.array_equal(codes, w_codes), what
    want = w_vals.astype(dtype)
    assert vals.dtype == want.dtype and np.array_equal(vals.view(np.uint8), want.view(np.uint8)), what
    return rp, codes, vals, tot


def _rows_ok(rp, codes, vals):
    n = len(rp) - 1
    for i in range(n):
        row = codes[int(rp[i]):int(rp[i + 1])].astype(np.int64)
        assert np.all(np.diff(row) > 0), f"row {i} not ascending"
    assert np.all(vals > 0)


@pytest.mark.parametrize("k", range(1, 13))
@pytest.mark.parametrize("canonical", [1, 0])
@pytest.mark.parametrize("norm,code", COMBOS)
def test_sparse_equals_dense_rows(k, canonical, norm, code):
    rng = np.random.default_rng(k * 100 + canonical * 10 + norm * 3 + code)
    nseq = 24 if k <= 9 else 6
    lens = [0, k - 1, k, 150, T + 7, 3 * T + 11] + list(rng.integers(0, 2500, size=nseq - 6))
    bases, offsets = random_batch(rng, lens, noise=0.02, n_runs=0.3)
    dtype = DT[code]
    rp, codes, vals, tot = check_against_ref(bases, offsets, k, canonical, norm, dtype, what=f"k={k}")
    _rows_ok(rp, codes, vals)
    oc = OligoComputer(k)
    dense = oc.vectorise_packed(bases, offsets, norm_mode=norm, mins=bool(canonical), dtype=dtype)
    pos_map = oc.kmer_pos_maps()[0] if canonical else None
    oc.close()
    got = scatter(rp, codes, vals, dense.shape[1], pos_map, dtype=dtype)
    assert np.array_equal(got.view(np.uint8), dense.view(np.uint8))
    if k <= 8:
        want, _ = oracle.vectorise_batch(bases, offsets, k, bool(canonical), norm)
        assert np.array_equal(got.view(np.uint8), want.astype(dtype).view(np.uint8))


@pytest.mark.parametrize("k", [13, 16, 17, 21, 30, 31])
@pytest.mark.parametrize("canonical", [1, 0])
@pytest.mark.parametrize("norm,code", [(0, 0), (1, 1), (2, 2)])
def test_sparse_large_k(k, canonical, norm, code):
    rng = np.random.default_rng(k * 7 + canonical + norm)
    lens = [0, k - 1, k, k + 1, 31, 300, T - 1, T, T + 1, 2 * T + 3] + list(rng.integers(0, 3000, size=20))
    bases, offsets = random_batch(rng, lens, noise=0.01, n_runs=0.2)
    # low-complexity and palindromic records: long runs of one key
    extra = [b"A" * 5000, b"ACGT" * 1500, b"AT" * 3000, b"GGCC" * 2500, (b"ACGT" * 8 + b"N") * 300]
    bases = np.concatenate([bases] + [np.frombuffer(e, np.uint8) for e in extra])
    offsets = np.concatenate([offsets, offsets[-1] + np.cumsum([len(e) for e in extra]).astype(np.uint64)])
    rp, codes, vals, _ = check_against_ref(bases, offsets, k, canonical, norm, DT[code], what=f"k={k}")
    _rows_ok(rp, codes, vals)


@pytest.mark.parametrize("k", [4, 16, 21, 31])
def test_sparse_tile_edges_and_long_merge(k):
    """Lengths around the tile size, reads laid across tile edges, and one 5 Mbp sequence (1221 tiles: 11 merge
    rounds with a trailing odd group)."""
    rng = np.random.default_rng(k)
    lens = [0, k - 1, k, T - 1, T, T + 1, 1, 0, 0, 2 * T - 1, 2 * T + 1, 150, 150, 150]
    lens += [T - 75] + [150] * 60                     # reads that straddle tile edges at various offsets
    lens += [5_000_000 + 17] + [T - 3, 1, 2, 3, 0, 5 * T]
    bases, offsets = random_batch(rng, lens, noise=0.005, n_runs=0.2)
    for canonical in (1, 0):
        check_against_ref(bases, offsets, k, canonical, 1, np.float32, what=f"k={k} canonical={canonical}")


def test_sparse_many_short_reads():
    rng = np.random.default_rng(5)
    bases, offsets = random_batch(rng, [150] * 100_000, noise=0.01, n_runs=0.05)
    check_against_ref(bases, offsets, 21, 1, 0, np.uint32)


def test_sparse_long_poly_a_large_divisor():
    """A poly-A record of 2^24 + 3 bases plus a mixed tail: divisors above 2^24 take the f64 path of make_out."""
    tail = np.frombuffer(b"ACGTTGCAAGGCTTAACCGGTTAA" * 40, np.uint8)
    rec = np.concatenate([np.full((1 << 24) + 3, ord("A"), np.uint8), tail])
    bases = np.concatenate([rec, np.frombuffer(b"ACGT" * 100, np.uint8)])
    offsets = np.array([0, len(rec), len(bases)], np.uint64)
    for k, canonical, norm, code in [(13, 1, 1, 1), (21, 0, 2, 1), (31, 1, 1, 2), (8, 1, 1, 1)]:
        check_against_ref(bases, offsets, k, canonical, norm, DT[code], what=f"k={k}")


# ---------------------------------------------------------------------------------------------------- device entry
torch = pytest.importorskip("torch")


def _dev_rows(tb, to, n, total, k, canonical=1, norm=0, code=0, cap=None, totals=True, stream=None, fence=64):
    """One device-entry call with every output fenced by sentinels; returns numpy rows trimmed to min(nnz, cap)."""
    dev = tb.device
    dtype = {0: torch.int32, 1: torch.float32, 2: torch.float64}[code]
    big = max(1, int(total))
    cap = big if cap is None else cap
    sent = {torch.int32: -7, torch.float32: -7.5, torch.float64: -7.25}[dtype]
    rp = torch.full((n + 1 + 2 * fence,), -3, dtype=torch.int64, device=dev)
    tt = torch.full((n + 2 * fence,), -5, dtype=torch.int64, device=dev)
    cd = torch.full((cap + 2 * fence,), -9, dtype=torch.int64, device=dev)
    vl = torch.full((cap + 2 * fence,), sent, dtype=dtype, device=dev)
    st = stream or torch.cuda.current_stream(dev)
    st.wait_stream(torch.cuda.current_stream(dev))   # the fences were filled on the current stream
    L = _lib.load()

    def ptr(t):
        return t.data_ptr() + fence * t.element_size()
    with torch.cuda.stream(st):
        _lib.check(L.ktb_sparse_vectorise_device(tb.data_ptr() if total else None, to.data_ptr(), n, total, k, canonical,
                                                 norm, code, ptr(rp), ptr(cd) if cap else None,
                                                 ptr(vl) if cap else None, cap, ptr(tt) if totals else None,
                                                 st.cuda_stream))
    return rp, tt, cd, vl, cap, fence, st, sent


def _finish(res, n, totals=True):
    rp, tt, cd, vl, cap, fence, st, sent = res
    st.synchronize()
    rp, tt, cd, vl = (x.cpu().numpy() for x in (rp, tt, cd, vl))
    assert np.all(rp[:fence] == -3) and np.all(rp[fence + n + 1:] == -3)
    assert np.all(tt[:fence] == -5) and np.all(tt[fence + n:] == -5)
    if not totals:
        assert np.all(tt == -5)
    row_ptr = rp[fence:fence + n + 1].astype(np.uint64)
    nnz = int(row_ptr[-1])
    m = min(nnz, cap)
    assert np.all(cd[:fence] == -9) and np.all(cd[fence + m:] == -9)
    assert np.all(vl[:fence] == sent) and np.all(vl[fence + m:] == sent)
    return row_ptr, cd[fence:fence + m].astype(np.uint64), vl[fence:fence + m], tt[fence:fence + n].astype(np.uint64)


def test_sparse_device_entry_views_cap_and_totals():
    rng = np.random.default_rng(11)
    lens = [0, 20, 150, T + 9, 3000, 0, 40, 2 * T + 1, 7] + list(rng.integers(0, 900, size=40))
    bases, offsets = random_batch(rng, lens, noise=0.02, n_runs=0.2)
    k, norm, code = 17, 1, 1
    want = sparse_rows(bases, offsets, k, True, norm)
    wv = want[2].astype(np.float32)
    dev = torch.device("cuda", 0)
    tb = torch.from_numpy(bases).to(dev)
    to = torch.from_numpy(offsets.astype(np.int64)).to(dev)
    n = len(lens)
    nnz = int(want[0][-1])
    for cap, with_tot in [(nnz, True), (nnz // 3, False), (0, True), (None, False)]:
        rp, cd, vl, tt = _finish(_dev_rows(tb, to, n, len(bases), k, 1, norm, code, cap=cap, totals=with_tot), n, with_tot)
        assert np.array_equal(rp, want[0])
        m = len(cd)
        assert np.array_equal(cd, want[1][:m]) and np.array_equal(vl.view(np.uint32), wv[:m].view(np.uint32))
        if with_tot:
            assert np.array_equal(tt, want[3])
    # sub-batch views: offsets[0] > 0, absolute positions, total_bases = offsets[hi]
    for lo, hi in [(1, 5), (3, 20), (7, n), (10, 10)]:
        w = sparse_rows(bases, offsets[lo:hi + 1], k, True, norm)
        rp, cd, vl, tt = _finish(_dev_rows(tb, to[lo:], hi - lo, int(offsets[hi]), k, 1, norm, code), hi - lo)
        assert np.array_equal(rp, w[0]) and np.array_equal(cd, w[1]) and np.array_equal(tt, w[3])
        assert np.array_equal(vl.view(np.uint32), w[2].astype(np.float32).view(np.uint32))


def test_sparse_device_entry_past_2_pow_32():
    """One batch placed past 2^32 in a 4 GiB + 1 MiB buffer: 64-bit positions in the tile search and the pool."""
    rng = np.random.default_rng(12)
    lens = [300, T + 5, 0, 1000, 150, 2 * T]
    bases, offsets = random_batch(rng, lens, noise=0.01)
    torch.cuda.empty_cache()
    dev = torch.device("cuda", 0)
    base = 1 << 32
    buf = torch.zeros(base + (1 << 20), dtype=torch.uint8, device=dev)
    buf[base:base + len(bases)] = torch.from_numpy(bases).to(dev)
    to = torch.from_numpy((offsets + np.uint64(base)).astype(np.int64)).to(dev)
    k = 21
    rp, cd, vl, tt = _finish(_dev_rows(buf, to, len(lens), base + len(bases), k, 0, 0, 0, cap=len(bases)), len(lens))
    w = sparse_rows(bases, offsets, k, False, 0)
    assert np.array_equal(rp, w[0]) and np.array_equal(cd, w[1]) and np.array_equal(tt, w[3])
    assert np.array_equal(vl.view(np.uint32), w[2].astype(np.uint32))
    del buf
    torch.cuda.empty_cache()


def test_sparse_device_entry_two_streams_and_determinism():
    rng = np.random.default_rng(13)
    dev = torch.device("cuda", 0)
    a = random_batch(rng, list(rng.integers(0, 3000, size=300)) + [200_000], noise=0.01, n_runs=0.1)
    b = random_batch(rng, [150] * 5000 + [3 * T + 1], noise=0.01)
    ta = [torch.from_numpy(x.astype(np.int64) if x.dtype == np.uint64 else x).to(dev) for x in a]
    tb_ = [torch.from_numpy(x.astype(np.int64) if x.dtype == np.uint64 else x).to(dev) for x in b]
    s1, s2 = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    torch.cuda.synchronize()
    r1 = _dev_rows(ta[0], ta[1], len(a[1]) - 1, len(a[0]), 25, 1, 2, 2, stream=s1)
    r2 = _dev_rows(tb_[0], tb_[1], len(b[1]) - 1, len(b[0]), 12, 0, 1, 1, stream=s2)
    r3 = _dev_rows(ta[0], ta[1], len(a[1]) - 1, len(a[0]), 25, 1, 2, 2, stream=s2)
    g1, g2, g3 = _finish(r1, len(a[1]) - 1), _finish(r2, len(b[1]) - 1), _finish(r3, len(a[1]) - 1)
    for x, y in zip(g1, g3):
        assert np.array_equal(x.view(np.uint8), y.view(np.uint8))
    check_against_ref(*a, 25, 1, 2, np.float64, got=g1)
    check_against_ref(*b, 12, 0, 1, np.float32, got=g2)


def test_sparse_host_entry_chunks_equal_device_entry():
    """More than three host chunks (2^26 bases each) against one device-entry call over the whole batch."""
    rng = np.random.default_rng(14)
    lens = list(rng.integers(1000, 40_000, size=14_000))   # about 2.9e8 bases
    bases, offsets = random_batch(rng, lens, noise=0.01)
    assert offsets[-1] > 4 * (1 << 26)
    k = 21
    host = kmer_counts((bases, offsets), k, True, 0, np.uint32)
    dev = torch.device("cuda", 0)
    tb = torch.from_numpy(bases).to(dev)
    to = torch.from_numpy(offsets.astype(np.int64)).to(dev)
    got = _finish(_dev_rows(tb, to, len(lens), len(bases), k, 1, 0, 0, fence=4), len(lens))
    assert np.array_equal(host[0], got[0]) and np.array_equal(host[3], got[3])
    assert np.array_equal(host[1], got[1]) and np.array_equal(host[2], got[2].view(np.uint32))
    # and a sample of rows against the oracle restatement
    for i in rng.integers(0, len(lens), size=5):
        lo, hi = int(offsets[i]), int(offsets[i + 1])
        w = sparse_rows(bases[lo:hi], np.array([0, hi - lo], np.uint64), k, True, 0)
        assert np.array_equal(host[1][int(host[0][i]):int(host[0][i + 1])], w[1])


@pytest.mark.parametrize("k", [4, 7, 10])
@pytest.mark.parametrize("dtype", ["float32", "float64", "int32"])
def test_sparse_tensor_rank_columns_equal_dense_tensors(k, dtype):
    rng = np.random.default_rng(k)
    lens = [0, 3, 150, T + 1, 2000] + list(rng.integers(0, 1500, size=20))
    bases, offsets = random_batch(rng, lens, noise=0.02, n_runs=0.2)
    dev = torch.device("cuda", 0)
    tb = torch.from_numpy(bases).to(dev)
    to = torch.from_numpy(offsets.astype(np.int64)).to(dev)
    tdt = getattr(torch, dtype)
    norm = 0 if dtype == "int32" else 1
    csr = kmer_counts_tensors(tb, to, k, True, norm, tdt, columns="rank")
    oc = OligoComputer(k)
    dense = oc.vectorise_tensors(tb, to, norm, True, tdt)
    oc.close()
    assert torch.equal(csr.to_dense(), dense)
    code_csr = kmer_counts_tensors(tb, to, k, True, norm, tdt)
    assert tuple(code_csr.shape) == (len(lens), 4 ** k)
    assert torch.equal(code_csr.crow_indices(), csr.crow_indices())
    with pytest.raises(ValueError):
        kmer_counts_tensors(tb, to, k, False, norm, tdt, columns="rank")
