// device_scan.cuh — host helpers shared by the sparse rows (sparse.cu) and the k-mer counter (counter.cu): the u64
// exclusive scan and a bump allocator over one stream-ordered allocation.
#pragma once
#include "host_common.h"
#include "sparse_common.cuh"

#include <cuda_runtime.h>
#include <stdint.h>

namespace ktb {

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
