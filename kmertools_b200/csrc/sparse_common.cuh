// sparse_common.cuh — device helpers shared by the sparse rows (sparse_kernels.cuh) and the k-mer counter
// (count_kernels.cuh): binary searches over sorted u64 arrays and a block-wide exclusive scan.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace ktb {

constexpr int SP_LOOK = 32;                         // staged look-back bytes (>= 31 - 1)
constexpr int SP_MTHREADS = 256;                    // merge, count, write and scan kernels
constexpr int SP_WITEMS = 16;
constexpr int SP_WB = SP_MTHREADS * SP_WITEMS;      // entries per block of the count / write passes and of the scans

// largest s in [lo, hi) with a[s] <= pos, given a[lo] <= pos < a[hi]
__device__ __forceinline__ uint64_t sp_find(const uint64_t *a, uint64_t lo, uint64_t hi, uint64_t pos) {
    while (hi - lo > 1) {
        const uint64_t mid = lo + ((hi - lo) >> 1);
        if (a[mid] <= pos) lo = mid; else hi = mid;
    }
    return lo;
}

__device__ __forceinline__ uint64_t sp_lower_bound(const uint64_t *a, uint64_t n, uint64_t key) {
    uint64_t lo = 0;
    while (n > 0) {
        const uint64_t half = n >> 1;
        if (a[lo + half] < key) { lo += half + 1; n -= half + 1; } else n = half;
    }
    return lo;
}

__device__ __forceinline__ uint64_t sp_upper_bound(const uint64_t *a, uint64_t n, uint64_t key) {
    uint64_t lo = 0;
    while (n > 0) {
        const uint64_t half = n >> 1;
        if (a[lo + half] <= key) { lo += half + 1; n -= half + 1; } else n = half;
    }
    return lo;
}

// exclusive block-wide scan; s_warp holds NT / 32 entries; every thread must call it
template <int NT>
__device__ __forceinline__ unsigned long long sp_block_scan(unsigned long long v, unsigned long long *s_warp,
                                                            unsigned long long &total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned long long incl = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const unsigned long long t = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += t;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        unsigned long long w = lane < NT / 32 ? s_warp[lane] : 0ull;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const unsigned long long t = __shfl_up_sync(0xffffffffu, w, d);
            if (lane >= d) w += t;
        }
        if (lane < NT / 32) s_warp[lane] = w;
    }
    __syncthreads();
    const unsigned long long base = warp ? s_warp[warp - 1] : 0ull;
    total = s_warp[NT / 32 - 1];
    __syncthreads();
    return base + incl - v;
}

}  // namespace ktb
