// host_common.h — host plumbing shared by the C ABI entry points: error reporting of CUDA calls, the device checks, and
// the chunked pipeline of the entry points that run a device entry point over host buffers (ktb_sparse_vectorise,
// ktb_counter_add, ktb_counter_coverage): the offset checks, the cut into chunks of whole sequences and the stream and
// buffers a chunk is copied into.  Each of those entry points keeps its own loop: their overlap schemes differ
// (DESIGN.md §7).
#pragma once
#include "../../include/kmertools_b200.h"

#include <cuda_runtime.h>
#include <stdint.h>
#include <algorithm>
#include <cstdio>
#include <vector>

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

// step(e, what) keeps the first failure of a sequence of CUDA calls in rc; the calls after it still run (teardown).
struct FirstError {
    int &rc;
    void operator()(cudaError_t e, const char *what) {
        if (rc == KTB_OK && e != cudaSuccess) rc = cuda_fail(what, e);
    }
};

inline int check_device(int device) {
    const int ndev = ktb_device_count();
    if (ndev <= 0) return ktb_internal_fail(KTB_ERR_NODEVICE, "no CUDA device available (this library has no CPU path)");
    if (device < 0 || device >= ndev) return ktb_internal_fail(KTB_ERR_ARG, "device out of range");
    return KTB_OK;
}

// SMs of the current device
inline int sm_count(int *sms) {
    int dev = 0;
    CUP(cudaGetDevice(&dev));
    CUP(cudaDeviceGetAttribute(sms, cudaDevAttrMultiProcessorCount, dev));
    return KTB_OK;
}

// bases of one chunk of a host entry point (a longer single sequence is a chunk of its own)
constexpr uint64_t HOST_CHUNK_BASES = 1ull << 26;

// Checks the offsets[0..n] of a host batch (non-decreasing) and that bases is there when they span any base.
// counts32 also refuses a sequence of more than 2^32 - 1 windows of k bases, for rows whose counts are u32.
inline int check_offsets(const uint8_t *bases, const uint64_t *offsets, uint64_t n, int k, bool counts32) {
    char msg[160];
    for (uint64_t i = 0; i < n; ++i) {
        if (offsets[i + 1] < offsets[i]) {
            snprintf(msg, sizeof msg, "offsets must be non-decreasing (at %llu)", (unsigned long long)i);
            return ktb_internal_fail(KTB_ERR_ARG, msg);
        }
        const uint64_t len = offsets[i + 1] - offsets[i];
        if (counts32 && len >= (uint64_t)k && len - (uint64_t)k + 1 > 0xFFFFFFFFull) {
            snprintf(msg, sizeof msg, "sequence %llu has %llu windows; counts are 32-bit (at most 2^32 - 1 windows)",
                     (unsigned long long)i, (unsigned long long)(len - (uint64_t)k + 1));
            return ktb_internal_fail(KTB_ERR_ARG, msg);
        }
    }
    if (offsets[n] > offsets[0] && !bases) return ktb_internal_fail(KTB_ERR_ARG, "bases is NULL");
    return KTB_OK;
}

// sequences [i0, i0 + n) of a batch, whose bases are [b0, b0 + nb)
struct Chunk {
    uint64_t i0, n, b0, nb;
};

// The cut of a checked host batch into chunks of whole sequences, at most HOST_CHUNK_BASES bases each unless one
// sequence is longer, and the largest bases and sequences of one chunk.
struct ChunkPlan {
    const uint8_t *bases;
    const uint64_t *offsets;
    std::vector<uint64_t> cut{0};
    uint64_t max_bases = 0, max_n = 0;

    ChunkPlan(const uint8_t *b, const uint64_t *off, uint64_t n) : bases(b), offsets(off) {
        for (uint64_t i0 = 0; i0 < n;) {
            uint64_t i1 = i0 + 1;
            while (i1 < n && offsets[i1 + 1] - offsets[i0] <= HOST_CHUNK_BASES) ++i1;
            max_bases = std::max(max_bases, offsets[i1] - offsets[i0]);
            max_n = std::max(max_n, i1 - i0);
            cut.push_back(i1);
            i0 = i1;
        }
    }
    // the most windows of k bases in one chunk (a pass over the offsets that only the sparse rows need)
    uint64_t max_windows(int k) const {
        uint64_t most = 0;
        for (uint64_t ci = 0; ci < chunks(); ++ci) {
            uint64_t windows = 0;
            for (uint64_t i = cut[ci]; i < cut[ci + 1]; ++i) {
                const uint64_t len = offsets[i + 1] - offsets[i];
                windows += len >= (uint64_t)k ? len - (uint64_t)k + 1 : 0;
            }
            most = std::max(most, windows);
        }
        return most;
    }
    uint64_t chunks() const { return cut.size() - 1; }
    Chunk operator[](uint64_t ci) const {
        const uint64_t i0 = cut[ci], i1 = cut[ci + 1];
        return {i0, i1 - i0, offsets[i0], offsets[i1] - offsets[i0]};
    }
};

// One of the two stream / buffer sets of a chunked host entry point: a non-blocking stream, the bases and offsets of a
// chunk on the device, and page-locked offsets to rebase them in.  An entry point derives its own slot for the extra
// buffers of its outputs, and frees those after release().
struct ChunkSlot {
    cudaStream_t st = nullptr;
    uint8_t *bases = nullptr;
    uint64_t *offsets = nullptr, *h_offsets = nullptr;

    void alloc(const ChunkPlan &plan, FirstError &step) {
        step(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking), "cudaStreamCreate");
        step(cudaMalloc((void **)&bases, std::max<uint64_t>(plan.max_bases, 1)), "cudaMalloc(bases)");
        step(cudaMalloc((void **)&offsets, (plan.max_n + 1) * sizeof(uint64_t)), "cudaMalloc(offsets)");
        step(cudaHostAlloc((void **)&h_offsets, (plan.max_n + 1) * sizeof(uint64_t), cudaHostAllocDefault),
             "cudaHostAlloc(offsets)");
    }
    // enqueues the copy of chunk ci to the device on st; the last chunk on st must be done with h_offsets
    void copy_in(const ChunkPlan &plan, uint64_t ci, FirstError &step) {
        const Chunk ch = plan[ci];
        for (uint64_t i = 0; i <= ch.n; ++i) h_offsets[i] = plan.offsets[ch.i0 + i] - ch.b0;
        if (ch.nb)
            step(cudaMemcpyAsync(bases, plan.bases + ch.b0, ch.nb, cudaMemcpyHostToDevice, st), "cudaMemcpyAsync(bases)");
        step(cudaMemcpyAsync(offsets, h_offsets, (ch.n + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, st),
             "cudaMemcpyAsync(offsets)");
    }
    // waits for the stream (a failure reaches step), then frees the buffers and the stream
    void release(FirstError &step) {
        if (st) step(cudaStreamSynchronize(st), "cudaStreamSynchronize");
        cudaFree(bases);
        cudaFree(offsets);
        cudaFreeHost(h_offsets);
        if (st) cudaStreamDestroy(st);
    }
};

}  // namespace ktb
