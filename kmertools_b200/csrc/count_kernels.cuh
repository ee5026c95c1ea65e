// count_kernels.cuh — batch-wide k-mer counting (ktb_counter_*, DESIGN.md §4.6).
//
// One add of a batch to a counter's table, 1 <= k <= 31:
//   count_valid_kernel / count_keys_kernel : the base stream is cut into flat tiles of CT_T window-end positions, staged
//                          as sparse_tile_kernel stages them (SP_LOOK look-back bytes of the same sequence, a reset at each
//                          sequence start).  The first pass counts each tile's valid windows; after a scan of those counts
//                          the second pass computes the keys again and writes the valid ones densely, in position order.
//   count_upsweep_kernel / count_scatter_kernel : stable LSD radix sort of the keys alone, 8-bit digits over only the 2k
//                          key bits (ceil(2k / 8) passes).  Per pass: the digit histogram of every tile of RX_T keys, a scan
//                          of the digit-major [256][tiles] matrix, then each tile sorts itself stably by the digit in shared
//                          memory (two 4-bit splits) and writes every key to its digit's global offset.
//   count_rle_*            : run-length encoding of the sorted keys: heads are counted per block, scanned and written with
//                          their positions; a run's count is the next head's position minus its own.
//   count_merge_*          : merge of the batch's (key, count) runs into the accumulated table.  Every element finds its
//                          output slot with one binary search in the other list; a key present in both lists is summed
//                          into the table's copy and the batch's copy is dropped (a flag, a scan, a compaction).
// Sizes that depend on the data (valid windows, runs, merged keys) stay on the device: grids are sized from the bases of
// the batch, and kernels read the actual sizes and stop there.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "sparse_common.cuh"
#include "values.cuh"

namespace ktb {

constexpr int CT_T = 4096;                       // window-end positions per key tile
constexpr int CT_THREADS = 512;
constexpr int CT_ITEMS = CT_T / CT_THREADS;      // consecutive positions per thread
constexpr uint8_t CT_START = 8;                  // staged-code flag: a sequence starts at this position

constexpr int RX_T = 4096;                       // keys per radix tile
constexpr int RX_THREADS = 512;
constexpr int RX_ITEMS = RX_T / RX_THREADS;
constexpr int RX_UTHREADS = 256;                 // upsweep; one thread per digit
constexpr int RX_DIGITS = 256;
constexpr size_t RX_SM_TOTAL = 2ull * RX_T * 8 + 16ull * RX_THREADS * 2;   // sort double buffer + 4-bit counters

struct CountKeysParams {
    const uint8_t *bases;
    const uint64_t *offsets;                 // n + 1, absolute
    uint64_t n;
    uint32_t k;
    int canonical;
    unsigned long long *tile_valid;          // ntiles: valid windows of each tile (count pass)
    const unsigned long long *tile_base;     // ntiles + 1: exclusive scan of tile_valid (key pass)
    uint64_t *keys;
};

// Keys of the window ends [ts, te) of one tile, CT_ITEMS consecutive positions per thread; bit j of the result is set
// where item j is a valid window.  codes: shared [SP_LOOK + CT_T]; s_seq: shared [2].
__device__ __forceinline__ uint32_t ct_tile_keys(const CountKeysParams &p, uint64_t ts, uint64_t te, uint8_t *codes,
                                                 uint64_t *s_seq, uint64_t (&key)[CT_ITEMS]) {
    const int tid = threadIdx.x;
    if (tid == 0) {
        s_seq[0] = sp_find(p.offsets, 0, p.n, ts);
        s_seq[1] = sp_find(p.offsets, s_seq[0], p.n, te - 1);
    }
    __syncthreads();
    const uint64_t s0 = s_seq[0], s1 = s_seq[1];
    const uint64_t s0start = p.offsets[s0];
    for (int i = tid; i < SP_LOOK + CT_T; i += CT_THREADS) {
        uint32_t c = 4u;
        if (ts + i >= s0start + SP_LOOK && ts + i < te + SP_LOOK) c = nt4_code(p.bases[ts + i - SP_LOOK]);
        codes[i] = (uint8_t)c;
    }
    __syncthreads();
    // empty sequences share a start byte: their threads store the same value
    for (uint64_t s = s0 + 1 + tid; s <= s1; s += CT_THREADS) codes[SP_LOOK + (p.offsets[s] - ts)] |= CT_START;
    __syncthreads();

    // the reference's rolling update restarted k - 1 positions back (DESIGN.md §2)
    const uint32_t k = p.k;
    const uint64_t mask = (1ull << (2 * k)) - 1ull;
    const uint32_t shift = 2 * (k - 1);
    const int i0 = tid * CT_ITEMS;
    uint64_t f = 0, r = 0;
    uint32_t run = 0;
    for (int q = i0 - (int)(k - 1); q < i0; ++q) {
        const uint32_t c = codes[q + SP_LOOK];
        if (c & CT_START) run = 0;
        const uint32_t b = c & 7u;
        if (b < 4u) {
            f = ((f << 2) | b) & mask;
            r = (r >> 2) | ((uint64_t)(b ^ 3u) << shift);
            ++run;
        } else {
            run = 0;
        }
    }
    uint32_t valid = 0;
#pragma unroll
    for (int j = 0; j < CT_ITEMS; ++j) {
        const uint32_t c = codes[i0 + j + SP_LOOK];
        if (c & CT_START) run = 0;
        const uint32_t b = c & 7u;
        if (b < 4u) {
            f = ((f << 2) | b) & mask;
            r = (r >> 2) | ((uint64_t)(b ^ 3u) << shift);
            ++run;
        } else {
            run = 0;
        }
        key[j] = p.canonical ? min(f, r) : f;
        valid |= (uint32_t)(run >= k) << j;
    }
    return valid;
}

__global__ void __launch_bounds__(CT_THREADS) count_valid_kernel(const CountKeysParams p) {
    __shared__ __align__(16) uint8_t codes[SP_LOOK + CT_T];
    __shared__ uint64_t s_seq[2];
    __shared__ unsigned long long s_scan[CT_THREADS / 32];
    const uint64_t base0 = p.offsets[0], end = p.offsets[p.n];
    const uint64_t ts = base0 + (uint64_t)blockIdx.x * CT_T;
    if (ts >= end) {
        if (threadIdx.x == 0) p.tile_valid[blockIdx.x] = 0;
        return;
    }
    uint64_t key[CT_ITEMS];
    const uint32_t valid = ct_tile_keys(p, ts, min(ts + (uint64_t)CT_T, end), codes, s_seq, key);
    unsigned long long total;
    sp_block_scan<CT_THREADS>((unsigned long long)__popc(valid), s_scan, total);
    if (threadIdx.x == 0) p.tile_valid[blockIdx.x] = total;
}

__global__ void __launch_bounds__(CT_THREADS) count_keys_kernel(const CountKeysParams p) {
    __shared__ __align__(16) uint8_t codes[SP_LOOK + CT_T];
    __shared__ uint64_t s_keys[CT_T];
    __shared__ uint64_t s_seq[2];
    __shared__ unsigned long long s_scan[CT_THREADS / 32];
    const uint64_t base0 = p.offsets[0], end = p.offsets[p.n];
    const uint64_t ts = base0 + (uint64_t)blockIdx.x * CT_T;
    if (ts >= end) return;
    uint64_t key[CT_ITEMS];
    const uint32_t valid = ct_tile_keys(p, ts, min(ts + (uint64_t)CT_T, end), codes, s_seq, key);
    unsigned long long total;
    uint32_t at = (uint32_t)sp_block_scan<CT_THREADS>((unsigned long long)__popc(valid), s_scan, total);
#pragma unroll
    for (int j = 0; j < CT_ITEMS; ++j)
        if (valid >> j & 1u) s_keys[at++] = key[j];
    __syncthreads();
    uint64_t *out = p.keys + p.tile_base[blockIdx.x];
    for (uint32_t i = threadIdx.x; i < (uint32_t)total; i += CT_THREADS) out[i] = s_keys[i];
}

// ================================================================================================
// LSD radix sort of the keys, one 8-bit digit per pass
// ================================================================================================
struct RadixParams {
    const uint64_t *in;
    uint64_t *out;
    const unsigned long long *nkeys;         // device: keys to sort
    uint64_t ntiles;                         // grid bound: tiles of RX_T keys
    uint32_t shift;                          // bit of this pass's digit
    unsigned long long *hist;                // [RX_DIGITS][ntiles] (upsweep)
    const unsigned long long *off;           // exclusive scan of hist (scatter)
};

__global__ void __launch_bounds__(RX_UTHREADS) count_upsweep_kernel(const RadixParams p) {
    __shared__ uint32_t h[RX_DIGITS];
    h[threadIdx.x] = 0;
    __syncthreads();
    const uint64_t nk = *p.nkeys, a = (uint64_t)blockIdx.x * RX_T, e = min(a + RX_T, nk);
    for (uint64_t i = a + threadIdx.x; i < e; i += RX_UTHREADS) atomicAdd(&h[(p.in[i] >> p.shift) & 255u], 1u);
    __syncthreads();
    p.hist[(uint64_t)threadIdx.x * p.ntiles + blockIdx.x] = h[threadIdx.x];
}

__global__ void __launch_bounds__(RX_THREADS, 2) count_scatter_kernel(const RadixParams p) {
    extern __shared__ __align__(16) uint8_t sm[];
    uint64_t *keys = reinterpret_cast<uint64_t *>(sm);                    // [2][RX_T]
    uint16_t *cnt = reinterpret_cast<uint16_t *>(sm + 2ull * RX_T * 8);   // [16][RX_THREADS]
    __shared__ uint32_t s_start[RX_DIGITS];
    __shared__ unsigned long long s_scan[RX_THREADS / 32];
    const uint64_t nk = *p.nkeys, a = (uint64_t)blockIdx.x * RX_T;
    if (a >= nk) return;
    const uint32_t nv = (uint32_t)min((uint64_t)RX_T, nk - a);
    const int tid = threadIdx.x, i0 = tid * RX_ITEMS;
    // past the last key: all-ones digits, so a stable sort leaves them behind every valid key
    for (int i = tid; i < RX_T; i += RX_THREADS) keys[i] = (uint32_t)i < nv ? p.in[a + i] : ~0ull;
    __syncthreads();
    uint64_t kk[RX_ITEMS];
#pragma unroll
    for (int j = 0; j < RX_ITEMS; ++j) kk[j] = keys[i0 + j];
    // stable split by the digit's low then high 4 bits; the blocked arrangement keeps it stable
    int cur = 0;
    for (uint32_t b = 0; b < 8; b += 4) {
        uint32_t dg[RX_ITEMS];
#pragma unroll
        for (int d = 0; d < 16; ++d) cnt[d * RX_THREADS + tid] = 0;
#pragma unroll
        for (int j = 0; j < RX_ITEMS; ++j) {
            dg[j] = (uint32_t)(kk[j] >> (p.shift + b)) & 15u;
            ++cnt[dg[j] * RX_THREADS + tid];
        }
        __syncthreads();
        uint16_t *row = cnt + tid * 16;   // raking scan over the counters in (digit, thread) order
        unsigned long long sum = 0, total;
#pragma unroll
        for (int e = 0; e < 16; ++e) sum += row[e];
        uint32_t acc = (uint32_t)sp_block_scan<RX_THREADS>(sum, s_scan, total);
#pragma unroll
        for (int e = 0; e < 16; ++e) {
            const uint32_t v = row[e];
            row[e] = (uint16_t)acc;
            acc += v;
        }
        __syncthreads();
        uint64_t *o = keys + (cur ^ 1) * RX_T;
#pragma unroll
        for (int j = 0; j < RX_ITEMS; ++j) o[cnt[dg[j] * RX_THREADS + tid]++] = kk[j];
        __syncthreads();
        cur ^= 1;
        if (b == 0) {
#pragma unroll
            for (int j = 0; j < RX_ITEMS; ++j) kk[j] = o[i0 + j];
        }
    }
    const uint64_t *sk = keys + cur * RX_T;
    for (uint32_t i = tid; i < nv; i += RX_THREADS) {
        const uint32_t d = (uint32_t)(sk[i] >> p.shift) & 255u;
        if (i == 0 || ((uint32_t)(sk[i - 1] >> p.shift) & 255u) != d) s_start[d] = i;
    }
    __syncthreads();
    for (uint32_t i = tid; i < nv; i += RX_THREADS) {
        const uint32_t d = (uint32_t)(sk[i] >> p.shift) & 255u;
        p.out[p.off[(uint64_t)d * p.ntiles + blockIdx.x] + (i - s_start[d])] = sk[i];
    }
}

// ================================================================================================
// run-length encoding of the sorted keys, blocks of SP_WB entries
// ================================================================================================
struct RleParams {
    const uint64_t *keys;                    // sorted
    const unsigned long long *nkeys;
    unsigned long long *block_heads;         // per block (count pass)
    const unsigned long long *block_base;    // exclusive scan of block_heads (write pass); [nblocks] = runs
    uint64_t *rkey;                          // runs: key
    uint64_t *rstart;                        //       position of the head
};

__device__ __forceinline__ uint32_t ct_heads(const RleParams &p, uint64_t i0, uint64_t nk) {
    uint32_t h = 0;
#pragma unroll
    for (int j = 0; j < SP_WITEMS; ++j) {
        const uint64_t i = i0 + j;
        h |= (uint32_t)(i < nk && (i == 0 || p.keys[i] != p.keys[i - 1])) << j;
    }
    return h;
}

__global__ void __launch_bounds__(SP_MTHREADS) count_rle_heads_kernel(const RleParams p) {
    __shared__ unsigned long long s_scan[SP_MTHREADS / 32];
    const uint64_t i0 = (uint64_t)blockIdx.x * SP_WB + (uint64_t)threadIdx.x * SP_WITEMS;
    unsigned long long total;
    sp_block_scan<SP_MTHREADS>((unsigned long long)__popc(ct_heads(p, i0, *p.nkeys)), s_scan, total);
    if (threadIdx.x == 0) p.block_heads[blockIdx.x] = total;
}

__global__ void __launch_bounds__(SP_MTHREADS) count_rle_write_kernel(const RleParams p) {
    __shared__ unsigned long long s_scan[SP_MTHREADS / 32];
    const uint64_t i0 = (uint64_t)blockIdx.x * SP_WB + (uint64_t)threadIdx.x * SP_WITEMS;
    const uint32_t h = ct_heads(p, i0, *p.nkeys);
    unsigned long long total;
    uint64_t at = p.block_base[blockIdx.x] + sp_block_scan<SP_MTHREADS>((unsigned long long)__popc(h), s_scan, total);
#pragma unroll
    for (int j = 0; j < SP_WITEMS; ++j)
        if (h >> j & 1u) {
            p.rkey[at] = p.keys[i0 + j];
            p.rstart[at] = i0 + j;
            ++at;
        }
}

// rcnt[j] = rstart[j + 1] - rstart[j], the last run ending at nkeys
__global__ void __launch_bounds__(SP_MTHREADS) count_rle_len_kernel(const uint64_t *rstart, const unsigned long long *nruns,
                                                                    const unsigned long long *nkeys, uint64_t *rcnt) {
    const uint64_t nr = *nruns, nk = *nkeys;
    for (uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; j < nr; j += (uint64_t)gridDim.x * blockDim.x)
        rcnt[j] = (j + 1 < nr ? rstart[j + 1] : nk) - rstart[j];
}

// ================================================================================================
// merge of the batch runs (b) into the table (a); both sorted, keys distinct within each list
// ================================================================================================
struct MergeParams {
    const uint64_t *akey, *acnt;
    uint64_t na;
    const uint64_t *bkey, *bcnt;
    const unsigned long long *nb;            // device
    uint64_t nb_bound;                       // entries of dup the scan covers
    unsigned long long *dup;                 // nb_bound: 1 where b's key is in a
    const unsigned long long *D;             // nb_bound + 1: exclusive scan of dup
    uint64_t *okey, *ocnt;
    const unsigned long long *nkeys;         // valid windows of the batch
    unsigned long long *sizes;               // out: [0] valid windows, [1] keys of the merged table
};

__global__ void __launch_bounds__(SP_MTHREADS) count_merge_dup_kernel(const MergeParams p) {
    const uint64_t nb = *p.nb;
    for (uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; j < p.nb_bound;
         j += (uint64_t)gridDim.x * blockDim.x) {
        unsigned long long d = 0;
        if (j < nb) {
            const uint64_t key = p.bkey[j], ub = sp_upper_bound(p.akey, p.na, key);
            d = ub && p.akey[ub - 1] == key;
        }
        p.dup[j] = d;
    }
}

__global__ void __launch_bounds__(SP_MTHREADS) count_merge_write_kernel(const MergeParams p) {
    const uint64_t nb = *p.nb, total = p.na + nb;
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        p.sizes[0] = *p.nkeys;
        p.sizes[1] = total - p.D[nb];
    }
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (uint64_t)gridDim.x * blockDim.x) {
        if (i < p.na) {   // a table key: every batch key below it that the table lacks comes first
            const uint64_t key = p.akey[i], lb = sp_lower_bound(p.bkey, nb, key);
            uint64_t c = p.acnt[i];
            if (lb < nb && p.bkey[lb] == key) c += p.bcnt[lb];
            const uint64_t o = i + lb - p.D[lb];
            p.okey[o] = key;
            p.ocnt[o] = c;
        } else {          // a batch key the table lacks: after every table key below it
            const uint64_t j = i - p.na;
            if (p.D[j + 1] != p.D[j]) continue;
            const uint64_t key = p.bkey[j], o = j - p.D[j] + sp_upper_bound(p.akey, p.na, key);
            p.okey[o] = key;
            p.ocnt[o] = p.bcnt[j];
        }
    }
}

}  // namespace ktb
