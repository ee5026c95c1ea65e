// coverage_kernels.cuh — per-read k-mer coverage histograms against a counter's table (ktb_counter_coverage*,
// DESIGN.md §4.7).
//
//   cov_dir_kernel   : a directory over the top b bits of the 2k-bit key of the sorted table: dir[p] = first index whose
//                      key has prefix >= p, dir[2^b] = nkeys.  One pass over the table: entry i fills the directory slots
//                      between the prefix of key i - 1 (exclusive) and its own (inclusive).  A lane writes a gap of up to
//                      32 slots itself; the warp writes a longer gap (a skewed table) together, 32 slots at a time.
//   cov_hist_kernel  : flat CT_T-position tiles of the batch, staged and keyed by ct_tile_keys (count_kernels.cuh).
//                      Every valid window looks up its abundance a (dir[p], dir[p + 1], then a binary search of at most
//                      2k - b probes inside that bucket; 0 when the key is absent) and adds 1 to bin
//                      min(a / bin_size, bin_count - 1) of its sequence.  The sequence of each piece of the tile (the part
//                      of one sequence inside it) is found once, by sp_find at the piece's start flag; per window it is a
//                      shared-memory read.  Windows of a warp that share (sequence, bin) are summed by __match_any_sync
//                      and added by one atomic.
//   cov_write_kernel : one warp per row: the row's sum is its total (every valid window is in one bin), then every bin
//                      is converted with norm_divisor / make_out (values.cuh), as the dense and sparse rows are.  For a
//                      4-byte output the u32 rows are the output buffer itself and are converted in place.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "count_kernels.cuh"

namespace ktb {

constexpr int COV_MAX_DIR_BITS = 30;            // directory of at most 2^30 + 1 entries (8 GiB)
constexpr uint32_t COV_MAX_BINS = 65536;
constexpr int COV_DIR_THREADS = 256;
constexpr int COV_WTHREADS = 256;

__global__ void __launch_bounds__(COV_DIR_THREADS) cov_dir_kernel(const uint64_t *keys, uint64_t nkeys, uint32_t shift,
                                                                  uint64_t nbuckets, uint64_t *dir) {
    const int lane = threadIdx.x & 31;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    // every warp runs the same number of iterations, so the whole warp takes part in each shuffle
    for (uint64_t base = (uint64_t)blockIdx.x * blockDim.x + (threadIdx.x & ~31u); base <= nkeys; base += stride) {
        const uint64_t i = base + lane;
        // slots (lo, hi] belong to entry i: the prefixes above key i - 1's, up to key i's (nbuckets past the last key)
        uint64_t lo = 0, hi = 0;
        if (i <= nkeys) {
            lo = i == 0 ? 0 : (keys[i - 1] >> shift) + 1;
            hi = i == nkeys ? nbuckets + 1 : (keys[i] >> shift) + 1;
        }
        const bool own = hi - lo <= 32;
        if (own)
            for (uint64_t q = lo; q < hi; ++q) dir[q] = i;
        for (uint32_t big = __ballot_sync(0xffffffffu, !own); big; big &= big - 1) {
            const int src = __ffs(big) - 1;
            const uint64_t a = __shfl_sync(0xffffffffu, lo, src), b = __shfl_sync(0xffffffffu, hi, src);
            for (uint64_t q = a + lane; q < b; q += 32) dir[q] = base + src;
        }
    }
}

struct CovParams {
    CountKeysParams kp;                      // bases, offsets, n, k, canonical (the other fields are unused)
    const uint64_t *tkey, *tcnt;             // the table
    uint64_t nkeys;
    const uint64_t *dir;                     // 2^(2k - shift) + 1 entries; unused when nkeys = 0
    uint32_t shift;                          // 2k - b: the prefix of a key is key >> shift
    uint32_t bin_size, bin_count;
    uint32_t *rows;                          // n x bin_count, zeroed
};

// abundance of one key: its count in the table, 0 when absent
__device__ __forceinline__ uint64_t cov_abundance(const CovParams &p, uint64_t key) {
    if (p.nkeys == 0) return 0;
    const uint64_t b = key >> p.shift;
    const uint64_t lo = p.dir[b], hi = p.dir[b + 1];
    const uint64_t at = lo + sp_lower_bound(p.tkey + lo, hi - lo, key);
    return at < hi && p.tkey[at] == key ? p.tcnt[at] : 0;
}

__global__ void __launch_bounds__(CT_THREADS) cov_hist_kernel(const CovParams p) {
    __shared__ __align__(16) uint8_t codes[SP_LOOK + CT_T];
    __shared__ uint64_t s_seq[2];
    __shared__ uint64_t s_piece[CT_T + 1];   // sequence of each piece of the tile
    __shared__ unsigned long long s_scan[CT_THREADS / 32];
    const uint64_t base0 = p.kp.offsets[0], end = p.kp.offsets[p.kp.n];
    const uint64_t ts = base0 + (uint64_t)blockIdx.x * CT_T;
    if (ts >= end) return;
    const uint64_t te = min(ts + (uint64_t)CT_T, end);
    uint64_t key[CT_ITEMS];
    const uint32_t valid = ct_tile_keys(p.kp, ts, te, codes, s_seq, key);

    // piece of each own position: 0 for s_seq[0], one more at every start flag; each piece's sequence is found once
    const int tid = threadIdx.x, i0 = tid * CT_ITEMS;
    uint32_t flags = 0;
#pragma unroll
    for (int j = 0; j < CT_ITEMS; ++j) flags |= (uint32_t)((codes[SP_LOOK + i0 + j] & CT_START) != 0) << j;
    unsigned long long total;
    uint32_t pi = (uint32_t)sp_block_scan<CT_THREADS>((unsigned long long)__popc(flags), s_scan, total);
    const uint64_t s0 = s_seq[0], s1 = s_seq[1];
    if (tid == 0) s_piece[0] = s0;
    uint32_t piece[CT_ITEMS];
#pragma unroll
    for (int j = 0; j < CT_ITEMS; ++j) {
        if (flags >> j & 1u) s_piece[++pi] = sp_find(p.kp.offsets, s0, s1 + 1, ts + i0 + j);
        piece[j] = pi;
    }
    __syncthreads();

    const int lane = tid & 31;
#pragma unroll
    for (int j = 0; j < CT_ITEMS; ++j) {
        uint64_t target = ~0ull;
        if (valid >> j & 1u) {
            const uint64_t a = cov_abundance(p, key[j]);
            const uint64_t q = a >> 32 ? a / p.bin_size : (uint64_t)((uint32_t)a / p.bin_size);
            const uint32_t bin = (uint32_t)min(q, (uint64_t)(p.bin_count - 1));
            target = s_piece[piece[j]] * p.bin_count + bin;
        }
        const uint32_t same = __match_any_sync(0xffffffffu, target);
        if (target != ~0ull && lane == __ffs(same) - 1) atomicAdd(&p.rows[target], (uint32_t)__popc(same));
    }
}

// rows (u32 counts) -> out (out_dtype) and totals; rows may alias out when OUT is 4 bytes wide
template <int OUT>
__global__ void __launch_bounds__(COV_WTHREADS) cov_write_kernel(const uint32_t *rows, void *out, uint64_t *totals,
                                                                 uint64_t n, uint32_t bin_count, int norm_mode) {
    using T = typename OutT<OUT>::type;
    T *o = reinterpret_cast<T *>(out);
    const bool norm = norm_mode != NORM_COUNTS;
    const int lane = threadIdx.x & 31;
    const uint64_t warps = (uint64_t)gridDim.x * (COV_WTHREADS / 32);
    for (uint64_t s = (uint64_t)blockIdx.x * (COV_WTHREADS / 32) + (threadIdx.x >> 5); s < n; s += warps) {
        const uint32_t *r = rows + s * bin_count;
        unsigned long long t = 0;
        for (uint32_t b = lane; b < bin_count; b += 32) t += r[b];
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) t += __shfl_xor_sync(0xffffffffu, t, d);
        if (totals && lane == 0) totals[s] = t;
        if (OUT == OUT_U32) continue;
        const uint64_t dv = norm_divisor(t, norm_mode, 1);
        const float dF = (float)dv;
        const float rinv = __frcp_rn(dF);
        T *w = o + s * bin_count;
        for (uint32_t b = lane; b < bin_count; b += 32)
            w[b] = make_out<OUT>(r[b], norm, dv < (1ull << 24), dF, rinv, (double)dv);
    }
}

}  // namespace ktb
