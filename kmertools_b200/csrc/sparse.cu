// sparse.cu — C ABI of the sparse per-sequence k-mer count rows (CSR): ktb_sparse_vectorise_device enqueues the
// kernels of sparse_kernels.cuh; ktb_sparse_vectorise runs it over host buffers in chunks of sequences.
#include "device_guard.h"
#include "device_scan.cuh"
#include "sparse_kernels.cuh"

#include <cuda_runtime.h>
#include <stdint.h>
#include <algorithm>
#include <cstdio>

namespace {

using namespace ktb;

int check_args(int k, int canonical, int norm_mode, int out_dtype) {
    char msg[128];
    if (k < 1 || k > KTB_MAX_SPARSE_K) {
        snprintf(msg, sizeof msg, "k must be in 1..%d for sparse rows (got %d)", KTB_MAX_SPARSE_K, k);
        return ktb_internal_fail(KTB_ERR_ARG, msg);
    }
    if (canonical != 0 && canonical != 1) return ktb_internal_fail(KTB_ERR_ARG, "canonical must be 0 or 1");
    if (norm_mode < KTB_NORM_COUNTS || norm_mode > KTB_NORM_PY) return ktb_internal_fail(KTB_ERR_ARG, "unknown norm_mode");
    if (out_dtype < KTB_OUT_U32 || out_dtype > KTB_OUT_F64) return ktb_internal_fail(KTB_ERR_ARG, "unknown out_dtype");
    if (out_dtype == KTB_OUT_U32 && norm_mode != KTB_NORM_COUNTS)
        return ktb_internal_fail(KTB_ERR_ARG, "KTB_OUT_U32 needs KTB_NORM_COUNTS");
    return KTB_OK;
}

}  // namespace

__attribute__((visibility("hidden"))) int ktb::scan_u64(const unsigned long long *in, uint64_t n,
                                                         unsigned long long *out, unsigned long long *bsum,
                                                         cudaStream_t st) {
    if (n == 0) {
        CUP(cudaMemsetAsync(out, 0, sizeof(uint64_t), st));
        return KTB_OK;
    }
    const uint64_t nb = div_up(n, SP_WB);
    sparse_scan_reduce_kernel<<<(unsigned)nb, SP_MTHREADS, 0, st>>>(in, n, bsum);
    sparse_scan_top_kernel<<<1, 1024, 0, st>>>(bsum, nb, out + n);
    sparse_scan_down_kernel<<<(unsigned)nb, SP_MTHREADS, 0, st>>>(in, n, bsum, out);
    CUP(cudaGetLastError());
    return KTB_OK;
}

int ktb_sparse_vectorise_device(const uint8_t *d_bases, const uint64_t *d_offsets, uint64_t n, uint64_t total_bases,
                                int k, int canonical, int norm_mode, int out_dtype, uint64_t *d_row_ptr,
                                uint64_t *d_codes, void *d_values, uint64_t cap, uint64_t *d_totals, void *stream) {
    if (int rc = check_args(k, canonical, norm_mode, out_dtype)) return rc;
    if (!d_offsets || !d_row_ptr) return ktb_internal_fail(KTB_ERR_ARG, "d_offsets / d_row_ptr is NULL");
    if (cap > 0 && (!d_codes || !d_values)) return ktb_internal_fail(KTB_ERR_ARG, "output arrays are NULL with cap > 0");
    if (total_bases > 0 && !d_bases) return ktb_internal_fail(KTB_ERR_ARG, "d_bases is NULL");
    cudaStream_t st = (cudaStream_t)stream;
    if (n == 0) {
        CUP(cudaMemsetAsync(d_row_ptr, 0, sizeof(uint64_t), st));
        return KTB_OK;
    }
    if (total_bases == 0) {   // every sequence is empty
        CUP(cudaMemsetAsync(d_row_ptr, 0, (n + 1) * sizeof(uint64_t), st));
        if (d_totals) CUP(cudaMemsetAsync(d_totals, 0, n * sizeof(uint64_t), st));
        return KTB_OK;
    }
    const uint64_t ntiles = div_up(total_bases, SP_T);
    if (ntiles > 0x7fffffffull) return ktb_internal_fail(KTB_ERR_ARG, "batch too large for one call");
    const uint64_t pool = ntiles * SP_T;
    const uint64_t nblocks = div_up(total_bases, SP_WB);   // the lists hold at most one entry per window
    const uint64_t nbsum = std::max(div_up(n, SP_WB), div_up(nblocks, SP_WB));

    int sms = 148;
    if (int rc = sm_count(&sms)) return rc;

    Carve c;
    auto layout = [&](SparseParams &p, SparseOutParams &o, unsigned long long *&V, unsigned long long *&bsum,
                      unsigned long long *&bbase) {
        p.pkey = c.take<uint64_t>(2 * pool);
        p.pcnt = c.take<uint32_t>(2 * pool);
        p.tot = c.take<unsigned long long>(n);
        p.len = c.take<unsigned long long>(n);
        p.nnz = c.take<unsigned long long>(n);
        p.loc = c.take<uint64_t>(n);
        p.desc = c.take<SparseDesc>(ntiles);
        p.gsize = c.take<uint64_t>(4 * ntiles);
        V = c.take<unsigned long long>(n + 1);
        o.block_nnz = c.take<unsigned long long>(nblocks);
        bbase = c.take<unsigned long long>(nblocks + 1);
        bsum = c.take<unsigned long long>(nbsum);
    };
    SparseParams p{};
    SparseOutParams o{};
    unsigned long long *V, *bsum, *bbase;
    layout(p, o, V, bsum, bbase);   // sizes only
    const size_t bytes = c.used;
    CUP(cudaMallocAsync((void **)&c.base, bytes, st));
    c.used = 0;
    layout(p, o, V, bsum, bbase);

    p.bases = d_bases;
    p.offsets = d_offsets;
    p.n = n;
    p.ntiles = ntiles;
    p.pool = pool;
    p.k = (uint32_t)k;
    p.canonical = canonical;
    int rc = KTB_OK;
    FirstError step{rc};
    step(cudaMemsetAsync(p.tot, 0, 3 * ((n * 8 + 255) & ~(size_t)255), st), "cudaMemsetAsync(per-sequence counters)");
    step(cudaMemsetAsync(p.desc, 0xFF, ntiles * sizeof(SparseDesc), st), "cudaMemsetAsync(tile descriptors)");
    step(cudaFuncSetAttribute(sparse_tile_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SP_SM_TOTAL),
         "cudaFuncSetAttribute(sparse_tile_kernel)");
    if (rc == KTB_OK) {
        sparse_tile_kernel<<<(unsigned)ntiles, SP_THREADS, SP_SM_TOTAL, st>>>(p);
        const unsigned mgrid = (unsigned)std::min<uint64_t>(ntiles, (uint64_t)sms * 8);
        for (uint32_t r = 1, rounds = sp_rounds(ntiles); r <= rounds; ++r)
            sparse_merge_kernel<<<mgrid, SP_MTHREADS, 0, st>>>(p, r);
        step(cudaGetLastError(), "sparse_tile_kernel / sparse_merge_kernel");
    }
    if (rc == KTB_OK) rc = scan_u64(p.len, n, V, bsum, st);
    if (rc == KTB_OK) rc = scan_u64(p.nnz, n, (unsigned long long *)d_row_ptr, bsum, st);
    if (rc == KTB_OK) {
        o.V = (const uint64_t *)V;
        o.loc = p.loc;
        o.tot = p.tot;
        o.pkey = p.pkey;
        o.pcnt = p.pcnt;
        o.n = n;
        o.nblocks = nblocks;
        o.block_base = bbase;
        o.codes = d_codes;
        o.values = d_values;
        o.cap = cap;
        o.norm_mode = norm_mode;
        o.canonical = canonical;
        const unsigned wgrid = (unsigned)std::min<uint64_t>(nblocks, (uint64_t)sms * 8);
        if (cap > 0) {
            sparse_count_kernel<<<wgrid, SP_MTHREADS, 0, st>>>(o);
            step(cudaGetLastError(), "sparse_count_kernel");
            if (rc == KTB_OK) rc = scan_u64(o.block_nnz, nblocks, bbase, bsum, st);
            if (rc == KTB_OK) {
                if (out_dtype == KTB_OUT_U32) sparse_write_kernel<KTB_OUT_U32><<<wgrid, SP_MTHREADS, 0, st>>>(o);
                else if (out_dtype == KTB_OUT_F32) sparse_write_kernel<KTB_OUT_F32><<<wgrid, SP_MTHREADS, 0, st>>>(o);
                else sparse_write_kernel<KTB_OUT_F64><<<wgrid, SP_MTHREADS, 0, st>>>(o);
                step(cudaGetLastError(), "sparse_write_kernel");
            }
        }
    }
    if (rc == KTB_OK && d_totals)
        step(cudaMemcpyAsync(d_totals, p.tot, n * sizeof(uint64_t), cudaMemcpyDeviceToDevice, st), "cudaMemcpyAsync(totals)");
    const cudaError_t ef = cudaFreeAsync(c.base, st);
    if (rc == KTB_OK && ef != cudaSuccess) rc = cuda_fail("cudaFreeAsync(scratch)", ef);
    return rc;
}

int ktb_sparse_vectorise(const uint8_t *bases, const uint64_t *offsets, uint64_t n, int k, int canonical,
                         int norm_mode, int out_dtype, int device, uint64_t *row_ptr, uint64_t *codes, void *values,
                         uint64_t cap, uint64_t *totals) {
    if (int rc = check_args(k, canonical, norm_mode, out_dtype)) return rc;
    if (!offsets || !row_ptr) return ktb_internal_fail(KTB_ERR_ARG, "offsets / row_ptr is NULL");
    if (cap > 0 && (!codes || !values)) return ktb_internal_fail(KTB_ERR_ARG, "output arrays are NULL with cap > 0");
    if (int rc = check_offsets(bases, offsets, n, k, true)) return rc;
    if (int rc = check_device(device)) return rc;
    ktb::DeviceGuard device_guard(device);
    CUP(device_guard.err);
    if (n == 0) {
        row_ptr[0] = 0;
        return KTB_OK;
    }
    const ChunkPlan plan(bases, offsets, n);
    const uint64_t max_windows = std::max<uint64_t>(plan.max_windows(k), 1);
    const size_t esize = out_dtype == KTB_OUT_F64 ? 8 : 4;

    // Two slots.  Everything of chunk c + 1 is enqueued (bases in, kernels, row_ptr and totals out to page-locked
    // staging) before the host waits for chunk c, so the copy-out of chunk c's codes and values into the caller's
    // memory runs while chunk c + 1 computes on the other stream.
    struct Slot : ChunkSlot {
        uint64_t *row_ptr = nullptr, *codes = nullptr, *totals = nullptr;
        void *values = nullptr;
        uint64_t *h_row_ptr = nullptr, *h_totals = nullptr;   // page-locked staging
    } slot[2];
    int rc = KTB_OK;
    FirstError step{rc};
    for (Slot &s : slot) {
        s.alloc(plan, step);
        step(cudaMalloc((void **)&s.row_ptr, (plan.max_n + 1) * sizeof(uint64_t)), "cudaMalloc(row_ptr)");
        step(cudaMalloc((void **)&s.totals, plan.max_n * sizeof(uint64_t)), "cudaMalloc(totals)");
        step(cudaMalloc((void **)&s.codes, max_windows * sizeof(uint64_t)), "cudaMalloc(codes)");
        step(cudaMalloc(&s.values, max_windows * esize), "cudaMalloc(values)");
        step(cudaHostAlloc((void **)&s.h_row_ptr, (plan.max_n + 1) * sizeof(uint64_t), cudaHostAllocDefault),
             "cudaHostAlloc(row_ptr)");
        step(cudaHostAlloc((void **)&s.h_totals, plan.max_n * sizeof(uint64_t), cudaHostAllocDefault),
             "cudaHostAlloc(totals)");
    }
    const uint64_t nchunks = plan.chunks();
    auto enqueue = [&](uint64_t ci) {
        Slot &s = slot[ci & 1];
        const Chunk ch = plan[ci];
        s.copy_in(plan, ci, step);
        if (rc == KTB_OK)
            rc = ktb_sparse_vectorise_device(s.bases, s.offsets, ch.n, ch.nb, k, canonical, norm_mode, out_dtype,
                                             s.row_ptr, s.codes, s.values, max_windows, s.totals, s.st);
        step(cudaMemcpyAsync(s.h_row_ptr, s.row_ptr, (ch.n + 1) * sizeof(uint64_t), cudaMemcpyDeviceToHost, s.st),
             "cudaMemcpyAsync(row_ptr)");
        if (totals)
            step(cudaMemcpyAsync(s.h_totals, s.totals, ch.n * sizeof(uint64_t), cudaMemcpyDeviceToHost, s.st),
                 "cudaMemcpyAsync(totals)");
    };
    uint64_t written = 0;   // entries of the rows before the current chunk
    if (rc == KTB_OK) enqueue(0);
    for (uint64_t ci = 0; ci < nchunks && rc == KTB_OK; ++ci) {
        if (ci + 1 < nchunks) enqueue(ci + 1);
        Slot &s = slot[ci & 1];
        step(cudaStreamSynchronize(s.st), "cudaStreamSynchronize");
        if (rc != KTB_OK) break;
        const Chunk ch = plan[ci];
        const uint64_t nnz = s.h_row_ptr[ch.n];
        for (uint64_t i = 0; i <= ch.n; ++i) row_ptr[ch.i0 + i] = written + s.h_row_ptr[i];
        if (totals) std::copy(s.h_totals, s.h_totals + ch.n, totals + ch.i0);
        const uint64_t ncopy = written >= cap ? 0 : std::min(nnz, cap - written);
        if (ncopy) {   // ordered on this slot's stream before its next chunk is copied in
            step(cudaMemcpyAsync(codes + written, s.codes, ncopy * sizeof(uint64_t), cudaMemcpyDeviceToHost, s.st),
                 "cudaMemcpyAsync(codes)");
            step(cudaMemcpyAsync((char *)values + written * esize, s.values, ncopy * esize, cudaMemcpyDeviceToHost, s.st),
                 "cudaMemcpyAsync(values)");
        }
        written += nnz;
    }
    for (Slot &s : slot) {
        s.release(step);
        cudaFree(s.row_ptr);
        cudaFree(s.totals);
        cudaFree(s.codes);
        cudaFree(s.values);
        cudaFreeHost(s.h_row_ptr);
        cudaFreeHost(s.h_totals);
    }
    return rc;
}
