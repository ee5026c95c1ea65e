// kmer_pairs.cu — KmerGenerator on the GPU: every valid window of one sequence as a (forward, reverse-complement)
// pair of 2-bit codes, in position order (kmer/src/kmer.rs:80-106; pybindings/src/kmer.rs:38-44).
//
// The serial iterator of the reference becomes data-parallel through its closed form (SURVEY.md §8a): a window
// ending at p is emitted iff its k bases are unambiguous, so a thread can restart the rolling update k-1 bases
// before its span without carrying state.  Three launches: count per block, scan of the block counts, write.
// Output-bound (16 bytes per k-mer against 1 byte per base), so the spans are short and re-derived rather
// than staged.
#include "device_guard.h"
#include "host_common.h"

#include <cuda_runtime.h>
#include <stdint.h>
#include <cstdio>

namespace {

using ktb::cuda_fail;

constexpr int PAIR_THREADS = 256;
constexpr int PAIR_SPAN = 16;                                  // window end positions per thread
constexpr uint64_t PAIR_BLOCK = (uint64_t)PAIR_THREADS * PAIR_SPAN;

// kmer/src/kmer.rs:6-15: 0..3 and ACGTU in either case are bases, everything else is ambiguous (4)
__device__ __forceinline__ uint32_t pair_nt4(uint32_t b) {
    if (b < 4u) return b;
    const uint32_t u = b & 0xDFu;
    if (u == 'A') return 0u;
    if (u == 'C') return 1u;
    if (u == 'G') return 2u;
    if (u == 'T' || u == 'U') return 3u;
    return 4u;
}

// windows ending in [p0, p1): the reference's rolling update restarted at p0-(k-1)
template <typename Emit>
__device__ __forceinline__ uint32_t pair_span(const uint8_t *seq, uint64_t p0, uint64_t p1, uint32_t k, Emit emit) {
    const uint64_t mask = (k >= 32u) ? ~0ull : ((1ull << (2 * k)) - 1ull);
    const uint32_t shift = 2 * (k - 1);
    uint64_t f = 0, r = 0;
    uint32_t run = 0, emitted = 0;
    for (uint64_t p = (p0 >= k - 1) ? p0 - (k - 1) : 0; p < p1; ++p) {
        const uint32_t c = pair_nt4(seq[p]);
        if (c < 4u) {
            f = ((f << 2) | c) & mask;
            r = (r >> 2) | ((uint64_t)(c ^ 3u) << shift);
            ++run;
        } else {
            run = 0;
        }
        if (run == k) {
            --run;
            if (p >= p0) {
                emit(emitted, f, r);
                ++emitted;
            }
        }
    }
    return emitted;
}

__device__ __forceinline__ uint32_t block_exclusive_scan(uint32_t v, uint32_t *s_warp, uint32_t &block_total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t incl = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += t;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    uint32_t base = 0, total = 0;
    for (int w = 0; w < PAIR_THREADS / 32; ++w) {
        if (w < warp) base += s_warp[w];
        total += s_warp[w];
    }
    block_total = total;
    return base + incl - v;
}

__global__ void __launch_bounds__(PAIR_THREADS) pair_count_kernel(const uint8_t *seq, uint64_t len, uint32_t k,
                                                                 uint32_t *block_counts) {
    __shared__ uint32_t s_warp[PAIR_THREADS / 32];
    const uint64_t p0 = (uint64_t)blockIdx.x * PAIR_BLOCK + (uint64_t)threadIdx.x * PAIR_SPAN;
    const uint64_t p1 = min(len, p0 + PAIR_SPAN);
    uint32_t mine = 0;
    if (p0 < len) mine = pair_span(seq, p0, p1, k, [](uint32_t, uint64_t, uint64_t) {});
    uint32_t total;
    block_exclusive_scan(mine, s_warp, total);
    if (threadIdx.x == 0) block_counts[blockIdx.x] = total;
}

// exclusive scan of the block counts (one CTA walks the array in strips), total to *count
__global__ void __launch_bounds__(PAIR_THREADS) pair_scan_kernel(const uint32_t *block_counts, uint64_t nblocks,
                                                                uint64_t *block_base, unsigned long long *count) {
    __shared__ uint32_t s_warp[PAIR_THREADS / 32];
    uint64_t carry = 0;
    for (uint64_t b0 = 0; b0 < nblocks; b0 += PAIR_THREADS) {
        const uint64_t b = b0 + threadIdx.x;
        const uint32_t v = (b < nblocks) ? block_counts[b] : 0u;
        uint32_t total;
        const uint32_t excl = block_exclusive_scan(v, s_warp, total);
        if (b < nblocks) block_base[b] = carry + excl;
        carry += total;
        __syncthreads();
    }
    if (threadIdx.x == 0) *count = carry;
}

__global__ void __launch_bounds__(PAIR_THREADS) pair_write_kernel(const uint8_t *seq, uint64_t len, uint32_t k,
                                                                 const uint64_t *block_base, uint64_t cap,
                                                                 uint64_t *out_f, uint64_t *out_r) {
    __shared__ uint32_t s_warp[PAIR_THREADS / 32];
    const uint64_t p0 = (uint64_t)blockIdx.x * PAIR_BLOCK + (uint64_t)threadIdx.x * PAIR_SPAN;
    const uint64_t p1 = min(len, p0 + PAIR_SPAN);
    uint32_t mine = 0;
    if (p0 < len) mine = pair_span(seq, p0, p1, k, [](uint32_t, uint64_t, uint64_t) {});
    uint32_t total;
    const uint64_t at = block_base[blockIdx.x] + block_exclusive_scan(mine, s_warp, total);
    if (mine == 0) return;
    pair_span(seq, p0, p1, k, [&](uint32_t i, uint64_t f, uint64_t r) {
        if (at + i < cap) {
            out_f[at + i] = f;
            out_r[at + i] = r;
        }
    });
}

int check_k(int k) {
    if (k < 1 || k > 31) {
        char msg[96];
        snprintf(msg, sizeof msg, "k must be in 1..31 for k-mer pairs (got %d)", k);
        return ktb_internal_fail(KTB_ERR_ARG, msg);
    }
    return KTB_OK;
}

}  // namespace

int ktb_kmer_pairs_device(const uint8_t *d_seq, uint64_t len, int k, uint64_t *d_out_f, uint64_t *d_out_r,
                          uint64_t cap, uint64_t *d_count, void *stream) {
    if (int rc = check_k(k)) return rc;
    if (!d_count) return ktb_internal_fail(KTB_ERR_ARG, "d_count is NULL");
    if (cap > 0 && (!d_out_f || !d_out_r)) return ktb_internal_fail(KTB_ERR_ARG, "output arrays are NULL");
    if (len > 0 && !d_seq) return ktb_internal_fail(KTB_ERR_ARG, "d_seq is NULL");
    cudaStream_t st = (cudaStream_t)stream;
    if (len == 0) {
        CUP(cudaMemsetAsync(d_count, 0, sizeof(uint64_t), st));
        return KTB_OK;
    }
    const uint64_t nblocks = (len + PAIR_BLOCK - 1) / PAIR_BLOCK;
    if (nblocks > 0x7fffffffull) return ktb_internal_fail(KTB_ERR_ARG, "sequence too long for one call");
    uint32_t *block_counts = nullptr;
    uint64_t *block_base = nullptr;
    CUP(cudaMallocAsync((void **)&block_counts, nblocks * sizeof(uint32_t), st));
    CUP(cudaMallocAsync((void **)&block_base, nblocks * sizeof(uint64_t), st));
    pair_count_kernel<<<(unsigned)nblocks, PAIR_THREADS, 0, st>>>(d_seq, len, (uint32_t)k, block_counts);
    pair_scan_kernel<<<1, PAIR_THREADS, 0, st>>>(block_counts, nblocks, block_base, (unsigned long long *)d_count);
    if (cap > 0)
        pair_write_kernel<<<(unsigned)nblocks, PAIR_THREADS, 0, st>>>(d_seq, len, (uint32_t)k, block_base, cap,
                                                                     d_out_f, d_out_r);
    CUP(cudaGetLastError());
    CUP(cudaFreeAsync(block_counts, st));
    CUP(cudaFreeAsync(block_base, st));
    return KTB_OK;
}

int ktb_kmer_pairs(const uint8_t *seq, uint64_t len, int k, int device, uint64_t *out_f, uint64_t *out_r,
                   uint64_t cap, uint64_t *count) {
    if (int rc = check_k(k)) return rc;
    if (!count) return ktb_internal_fail(KTB_ERR_ARG, "count is NULL");
    if (cap > 0 && (!out_f || !out_r)) return ktb_internal_fail(KTB_ERR_ARG, "output arrays are NULL");
    if (len > 0 && !seq) return ktb_internal_fail(KTB_ERR_ARG, "seq is NULL");
    if (int rc = ktb::check_device(device)) return rc;
    ktb::DeviceGuard device_guard(device);
    CUP(device_guard.err);
    *count = 0;
    if (len < (uint64_t)k) return KTB_OK;
    const uint64_t max_pairs = len - (uint64_t)k + 1;
    const uint64_t dcap = cap < max_pairs ? cap : max_pairs;
    uint8_t *d_seq = nullptr;
    uint64_t *d_f = nullptr, *d_r = nullptr, *d_count = nullptr;
    int rc = KTB_OK;
    cudaError_t e = cudaMalloc((void **)&d_seq, len);
    if (e == cudaSuccess) e = cudaMalloc((void **)&d_count, sizeof(uint64_t));
    if (e == cudaSuccess && dcap) e = cudaMalloc((void **)&d_f, dcap * sizeof(uint64_t));
    if (e == cudaSuccess && dcap) e = cudaMalloc((void **)&d_r, dcap * sizeof(uint64_t));
    if (e == cudaSuccess) e = cudaMemcpy(d_seq, seq, len, cudaMemcpyHostToDevice);
    if (e != cudaSuccess) {
        rc = cuda_fail("k-mer pair buffers", e);
    } else {
        rc = ktb_kmer_pairs_device(d_seq, len, k, d_f, d_r, dcap, d_count, nullptr);
        uint64_t found = 0;
        if (rc == KTB_OK && (e = cudaMemcpy(&found, d_count, sizeof found, cudaMemcpyDeviceToHost)) != cudaSuccess)
            rc = cuda_fail("cudaMemcpy(count)", e);
        if (rc == KTB_OK) {
            *count = found;
            const uint64_t ncopy = found < dcap ? found : dcap;
            if (ncopy && (e = cudaMemcpy(out_f, d_f, ncopy * sizeof(uint64_t), cudaMemcpyDeviceToHost)) != cudaSuccess)
                rc = cuda_fail("cudaMemcpy(out_f)", e);
            if (rc == KTB_OK && ncopy &&
                (e = cudaMemcpy(out_r, d_r, ncopy * sizeof(uint64_t), cudaMemcpyDeviceToHost)) != cudaSuccess)
                rc = cuda_fail("cudaMemcpy(out_r)", e);
        }
    }
    cudaFree(d_seq);
    cudaFree(d_f);
    cudaFree(d_r);
    cudaFree(d_count);
    return rc;
}
