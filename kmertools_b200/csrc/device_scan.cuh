// device_scan.cuh — host helpers shared by the sparse rows (sparse.cu) and the k-mer counter (counter.cu): error
// reporting of CUDA calls, the u64 exclusive scan, and a bump allocator over one stream-ordered allocation.
#pragma once
#include "sparse_common.cuh"
#include "../../include/kmertools_b200.h"

#include <cuda_runtime.h>
#include <stdint.h>
#include <cstdio>

int ktb_internal_fail(int code, const char *msg);

namespace ktb {

inline int cuda_fail(const char *what, cudaError_t e) {
    char msg[256];
    snprintf(msg, sizeof msg, "%s failed: %s", what, cudaGetErrorString(e));
    return ktb_internal_fail(e == cudaErrorMemoryAllocation ? KTB_ERR_NOMEM : KTB_ERR_CUDA, msg);
}

#define CUP(call)                                                \
    do {                                                         \
        cudaError_t e_ = (call);                                 \
        if (e_ != cudaSuccess) return ktb::cuda_fail(#call, e_); \
    } while (0)

inline uint64_t div_up(uint64_t a, uint64_t b) { return (a + b - 1) / b; }

// exclusive scan of in[0..n) into out[0..n] (out[n] = sum) by the sparse_scan_* kernels; bsum: div_up(n, SP_WB)
// entries.  Defined in sparse.cu.
int scan_u64(const unsigned long long *in, uint64_t n, unsigned long long *out, unsigned long long *bsum,
             cudaStream_t st);

// bump allocator over one stream-ordered allocation
struct Carve {
    char *base = nullptr;
    size_t used = 0;
    template <typename T> T *take(uint64_t count) {
        T *p = reinterpret_cast<T *>(base ? base + used : nullptr);
        used += (count * sizeof(T) + 255) & ~(size_t)255;
        return p;
    }
};

}  // namespace ktb
