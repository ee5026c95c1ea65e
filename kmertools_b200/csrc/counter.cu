// counter.cu — C ABI of batch-wide k-mer counting (ktb_counter_*): a table of (key, u64 count) in ascending key order
// on one GPU, grown by adds of batches.  An add enqueues the kernels of count_kernels.cuh and waits for its stream once,
// at the end, to learn the new table size.  Coverage histograms (ktb_counter_coverage*) look each window of a batch up
// in that table through a directory built on first use (coverage_kernels.cuh).
#include "count_kernels.cuh"
#include "coverage_kernels.cuh"
#include "device_guard.h"
#include "device_scan.cuh"

#include <cuda_runtime.h>
#include <stdint.h>
#include <algorithm>
#include <cstdio>

using namespace ktb;

struct ktb_counter {
    int k = 0, canonical = 1, device = 0;
    uint64_t *keys = nullptr, *counts = nullptr;   // the table (stream-ordered allocations)
    uint64_t nkeys = 0, nwindows = 0;
    unsigned long long *h_sizes = nullptr;         // page-locked [2]: valid windows and table keys of the last add
    uint64_t *dir = nullptr;                       // coverage directory of this table (NULL until built; freed by an add)
    uint32_t dir_bits = 0;
};

namespace {

int check_k(int k, int canonical) {
    char msg[128];
    if (k < 1 || k > KTB_MAX_SPARSE_K) {
        snprintf(msg, sizeof msg, "k must be in 1..%d for the k-mer counter (got %d)", KTB_MAX_SPARSE_K, k);
        return ktb_internal_fail(KTB_ERR_ARG, msg);
    }
    if (canonical != 0 && canonical != 1) return ktb_internal_fail(KTB_ERR_ARG, "canonical must be 0 or 1");
    return KTB_OK;
}

// Enqueues the add of one batch (device buffers) on st and points the counter at the new table; the caller then waits
// for st and takes the sizes from h_sizes (finish_add).  Nothing is enqueued when the scratch or the new table does not
// fit: the counter is unchanged.  free_old = false leaves the old table allocated: the caller owns it from then on.
int enqueue_add(ktb_counter *c, const uint8_t *d_bases, const uint64_t *d_offsets, uint64_t n, uint64_t total,
                cudaStream_t st, bool free_old = true) {
    const uint64_t nt_k = div_up(total, CT_T);               // key tiles
    if (nt_k > 0x7fffffffull) return ktb_internal_fail(KTB_ERR_ARG, "batch too large for one add");
    const uint64_t W = total;                                // bound of the valid windows
    const uint64_t nt_r = div_up(W, RX_T);                   // radix tiles
    const uint64_t nblk = div_up(W, SP_WB);                  // run-length blocks
    const uint64_t space = c->k >= 31 ? ~0ull : (1ull << (2 * c->k));
    const uint64_t ncap = c->nkeys + std::min(W, space);     // bound of the merged table
    const uint64_t nbsum = div_up(std::max({nt_k, (uint64_t)RX_DIGITS * nt_r, nblk, W}), SP_WB);

    int sms = 148;
    if (int rc = sm_count(&sms)) return rc;

    Carve s;
    unsigned long long *tile_valid, *tile_base, *hist, *hoff, *bheads, *bbase, *R, *D, *bsum, *sizes;
    uint64_t *X, *Y;
    auto layout = [&] {
        tile_valid = s.take<unsigned long long>(nt_k);
        tile_base = s.take<unsigned long long>(nt_k + 1);
        X = s.take<uint64_t>(W);
        Y = s.take<uint64_t>(W);
        hist = s.take<unsigned long long>(RX_DIGITS * nt_r);
        hoff = s.take<unsigned long long>(RX_DIGITS * nt_r + 1);
        bheads = s.take<unsigned long long>(nblk);
        bbase = s.take<unsigned long long>(nblk + 1);
        R = s.take<unsigned long long>(W);
        D = s.take<unsigned long long>(W + 1);
        bsum = s.take<unsigned long long>(nbsum);
        sizes = s.take<unsigned long long>(2);
    };
    layout();   // sizes only
    const size_t bytes = s.used;
    uint64_t *okey = nullptr, *ocnt = nullptr;
    {
        cudaError_t e = cudaMallocAsync((void **)&s.base, bytes, st);
        if (e == cudaSuccess) e = cudaMallocAsync((void **)&okey, std::max<uint64_t>(ncap, 1) * 8, st);
        if (e == cudaSuccess) e = cudaMallocAsync((void **)&ocnt, std::max<uint64_t>(ncap, 1) * 8, st);
        if (e != cudaSuccess) {
            cudaFreeAsync(s.base, st);
            cudaFreeAsync(okey, st);
            cudaGetLastError();
            return cuda_fail("cudaMallocAsync(counter scratch and table)", e);
        }
    }
    s.used = 0;
    layout();

    int rc = KTB_OK;
    FirstError step{rc};
    // keys: count, scan, write
    CountKeysParams kp{d_bases, d_offsets, n, (uint32_t)c->k, c->canonical, tile_valid, tile_base, X};
    count_valid_kernel<<<(unsigned)nt_k, CT_THREADS, 0, st>>>(kp);
    step(cudaGetLastError(), "count_valid_kernel");
    if (rc == KTB_OK) rc = scan_u64(tile_valid, nt_k, tile_base, bsum, st);
    if (rc == KTB_OK) {
        count_keys_kernel<<<(unsigned)nt_k, CT_THREADS, 0, st>>>(kp);
        step(cudaGetLastError(), "count_keys_kernel");
    }
    const unsigned long long *nkeys = tile_base + nt_k;
    // sort: ceil(2k / 8) passes of 8 bits
    uint64_t *in = X, *out = Y;
    step(cudaFuncSetAttribute(count_scatter_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RX_SM_TOTAL),
         "cudaFuncSetAttribute(count_scatter_kernel)");
    for (uint32_t shift = 0; rc == KTB_OK && shift < 2u * (uint32_t)c->k; shift += 8) {
        RadixParams rp{in, out, nkeys, nt_r, shift, hist, hoff};
        count_upsweep_kernel<<<(unsigned)nt_r, RX_UTHREADS, 0, st>>>(rp);
        step(cudaGetLastError(), "count_upsweep_kernel");
        if (rc == KTB_OK) rc = scan_u64(hist, RX_DIGITS * nt_r, hoff, bsum, st);
        if (rc == KTB_OK) {
            count_scatter_kernel<<<(unsigned)nt_r, RX_THREADS, RX_SM_TOTAL, st>>>(rp);
            step(cudaGetLastError(), "count_scatter_kernel");
        }
        std::swap(in, out);
    }
    // run-length encoding: runs' keys to `out`, head positions to R, counts to `in` (the sorted keys are done by then)
    RleParams lp{in, nkeys, bheads, bbase, out, (uint64_t *)R};
    const unsigned grid = (unsigned)std::min<uint64_t>(std::max<uint64_t>(div_up(W, SP_MTHREADS), 1), (uint64_t)sms * 16);
    if (rc == KTB_OK) {
        count_rle_heads_kernel<<<(unsigned)nblk, SP_MTHREADS, 0, st>>>(lp);
        step(cudaGetLastError(), "count_rle_heads_kernel");
    }
    if (rc == KTB_OK) rc = scan_u64(bheads, nblk, bbase, bsum, st);
    const unsigned long long *nruns = bbase + nblk;
    if (rc == KTB_OK) {
        count_rle_write_kernel<<<(unsigned)nblk, SP_MTHREADS, 0, st>>>(lp);
        count_rle_len_kernel<<<grid, SP_MTHREADS, 0, st>>>((const uint64_t *)R, nruns, nkeys, in);
        step(cudaGetLastError(), "count_rle_write_kernel / count_rle_len_kernel");
    }
    // merge into the table
    MergeParams mp{c->keys, c->counts, c->nkeys, out, in, nruns, W, R, D, okey, ocnt, nkeys, sizes};
    if (rc == KTB_OK) {
        count_merge_dup_kernel<<<grid, SP_MTHREADS, 0, st>>>(mp);
        step(cudaGetLastError(), "count_merge_dup_kernel");
    }
    if (rc == KTB_OK) rc = scan_u64(R, W, D, bsum, st);
    if (rc == KTB_OK) {
        const unsigned mgrid = (unsigned)std::min<uint64_t>(std::max<uint64_t>(div_up(c->nkeys + W, SP_MTHREADS), 1),
                                                            (uint64_t)sms * 16);
        count_merge_write_kernel<<<mgrid, SP_MTHREADS, 0, st>>>(mp);
        step(cudaGetLastError(), "count_merge_write_kernel");
    }
    step(cudaMemcpyAsync(c->h_sizes, sizes, 2 * sizeof(uint64_t), cudaMemcpyDeviceToHost, st), "cudaMemcpyAsync(sizes)");
    step(cudaFreeAsync(s.base, st), "cudaFreeAsync(scratch)");
    if (rc != KTB_OK) {
        cudaFreeAsync(okey, st);
        cudaFreeAsync(ocnt, st);
        return rc;
    }
    if (free_old) {
        step(cudaFreeAsync(c->keys, st), "cudaFreeAsync(table)");
        step(cudaFreeAsync(c->counts, st), "cudaFreeAsync(table)");
    }
    if (c->dir) {   // it indexes the old table
        step(cudaFreeAsync(c->dir, st), "cudaFreeAsync(coverage directory)");
        c->dir = nullptr;
    }
    c->keys = okey;
    c->counts = ocnt;
    return rc;
}

int finish_add(ktb_counter *c, cudaStream_t st) {
    CUP(cudaStreamSynchronize(st));
    c->nwindows += c->h_sizes[0];
    c->nkeys = c->h_sizes[1];
    return KTB_OK;
}

// Directory bits for a table of nkeys keys: 2^b <= nkeys < 2^(b + 1), capped at 2k (a direct index) and at
// COV_MAX_DIR_BITS.
uint32_t dir_bits(uint64_t nkeys, int k) {
    const uint32_t b = nkeys ? 63u - (uint32_t)__builtin_clzll(nkeys) : 0u;
    return std::min<uint32_t>({b, 2u * (uint32_t)k, (uint32_t)COV_MAX_DIR_BITS});
}

// Builds the coverage directory of the current table on st and waits for it, once per table.  An empty table needs
// none.  A directory that does not fit is KTB_ERR_NOMEM and leaves the counter as it was.
int ensure_dir(ktb_counter *c, cudaStream_t st) {
    if (c->dir || c->nkeys == 0) return KTB_OK;
    const uint32_t b = dir_bits(c->nkeys, c->k);
    const uint64_t nb = 1ull << b;
    int sms = 148;
    if (int rc = sm_count(&sms)) return rc;
    uint64_t *dir = nullptr;
    if (const cudaError_t e = cudaMallocAsync((void **)&dir, (nb + 1) * sizeof(uint64_t), st)) {
        cudaGetLastError();   // not sticky: later calls must not see it
        return cuda_fail("cudaMallocAsync(coverage directory)", e);
    }
    const unsigned grid = (unsigned)std::min<uint64_t>(div_up(c->nkeys + 1, COV_DIR_THREADS), (uint64_t)sms * 8);
    cov_dir_kernel<<<grid, COV_DIR_THREADS, 0, st>>>(c->keys, c->nkeys, 2u * (uint32_t)c->k - b, nb, dir);
    cudaError_t e = cudaGetLastError();
    const cudaError_t es = cudaStreamSynchronize(st);
    if (e == cudaSuccess) e = es;
    if (e != cudaSuccess) {
        cudaFreeAsync(dir, st);
        return cuda_fail("cov_dir_kernel", e);
    }
    c->dir = dir;
    c->dir_bits = b;
    return KTB_OK;
}

int check_coverage_args(uint32_t bin_size, uint32_t bin_count, int norm_mode, int out_dtype) {
    if (bin_size < 1) return ktb_internal_fail(KTB_ERR_ARG, "bin_size must be at least 1");
    if (bin_count < 1 || bin_count > COV_MAX_BINS) return ktb_internal_fail(KTB_ERR_ARG, "bin_count must be in 1..65536");
    if (norm_mode != KTB_NORM_COUNTS && norm_mode != KTB_NORM_CLI)
        return ktb_internal_fail(KTB_ERR_ARG, "norm_mode must be KTB_NORM_COUNTS or KTB_NORM_CLI for coverage rows");
    if (out_dtype < KTB_OUT_U32 || out_dtype > KTB_OUT_F64) return ktb_internal_fail(KTB_ERR_ARG, "unknown out_dtype");
    if (out_dtype == KTB_OUT_U32 && norm_mode != KTB_NORM_COUNTS)
        return ktb_internal_fail(KTB_ERR_ARG, "KTB_OUT_U32 needs KTB_NORM_COUNTS");
    return KTB_OK;
}

// Enqueues the coverage rows of one batch (device buffers, arguments checked, directory built) on st.
int enqueue_coverage(const ktb_counter *c, const uint8_t *d_bases, const uint64_t *d_offsets, uint64_t n,
                     uint64_t total, uint32_t bin_size, uint32_t bin_count, int norm_mode, int out_dtype, void *d_out,
                     uint64_t *d_totals, cudaStream_t st) {
    const uint64_t nel = n * (uint64_t)bin_count;
    const size_t esize = out_dtype == KTB_OUT_F64 ? 8 : 4;
    if (total == 0) {   // every sequence is empty
        CUP(cudaMemsetAsync(d_out, 0, nel * esize, st));
        if (d_totals) CUP(cudaMemsetAsync(d_totals, 0, n * sizeof(uint64_t), st));
        return KTB_OK;
    }
    const uint64_t nt = div_up(total, CT_T);
    if (nt > 0x7fffffffull) return ktb_internal_fail(KTB_ERR_ARG, "batch too large for one call");
    int sms = 148;
    if (int rc = sm_count(&sms)) return rc;
    uint32_t *rows = (uint32_t *)d_out;   // 4-byte outputs are counted in place
    if (esize == 8)
        if (const cudaError_t e = cudaMallocAsync((void **)&rows, nel * sizeof(uint32_t), st)) {
            cudaGetLastError();
            return cuda_fail("cudaMallocAsync(coverage rows)", e);
        }
    int rc = KTB_OK;
    FirstError step{rc};
    step(cudaMemsetAsync(rows, 0, nel * sizeof(uint32_t), st), "cudaMemsetAsync(coverage rows)");
    CovParams p{};
    p.kp.bases = d_bases;
    p.kp.offsets = d_offsets;
    p.kp.n = n;
    p.kp.k = (uint32_t)c->k;
    p.kp.canonical = c->canonical;
    p.tkey = c->keys;
    p.tcnt = c->counts;
    p.nkeys = c->nkeys;
    p.dir = c->dir;
    p.shift = 2u * (uint32_t)c->k - c->dir_bits;
    p.bin_size = bin_size;
    p.bin_count = bin_count;
    p.rows = rows;
    if (rc == KTB_OK) {
        cov_hist_kernel<<<(unsigned)nt, CT_THREADS, 0, st>>>(p);
        step(cudaGetLastError(), "cov_hist_kernel");
    }
    if (rc == KTB_OK) {
        const unsigned grid = (unsigned)std::min<uint64_t>(div_up(n, COV_WTHREADS / 32), (uint64_t)sms * 16);
        if (out_dtype == KTB_OUT_U32) cov_write_kernel<OUT_U32><<<grid, COV_WTHREADS, 0, st>>>(rows, d_out, d_totals, n, bin_count, norm_mode);
        else if (out_dtype == KTB_OUT_F32) cov_write_kernel<OUT_F32><<<grid, COV_WTHREADS, 0, st>>>(rows, d_out, d_totals, n, bin_count, norm_mode);
        else cov_write_kernel<OUT_F64><<<grid, COV_WTHREADS, 0, st>>>(rows, d_out, d_totals, n, bin_count, norm_mode);
        step(cudaGetLastError(), "cov_write_kernel");
    }
    if (esize == 8) step(cudaFreeAsync(rows, st), "cudaFreeAsync(coverage rows)");
    return rc;
}

}  // namespace

extern "C" {

int ktb_counter_create(int k, int canonical, int device, ktb_counter **out) {
    if (!out) return ktb_internal_fail(KTB_ERR_ARG, "out is NULL");
    *out = nullptr;
    if (int rc = check_k(k, canonical)) return rc;
    if (device < 0) return ktb_internal_fail(KTB_ERR_ARG, "device out of range");
    if (int rc = check_device(device)) return rc;
    ktb::DeviceGuard device_guard(device);
    CUP(device_guard.err);
    ktb_counter *c = new ktb_counter();
    c->k = k;
    c->canonical = canonical;
    c->device = device;
    const cudaError_t e = cudaHostAlloc((void **)&c->h_sizes, 2 * sizeof(uint64_t), cudaHostAllocDefault);
    if (e != cudaSuccess) {
        delete c;
        return cuda_fail("cudaHostAlloc(sizes)", e);
    }
    *out = c;
    return KTB_OK;
}

void ktb_counter_destroy(ktb_counter *c) {
    if (!c) return;
    ktb::DeviceGuard device_guard(c->device);
    cudaFree(c->keys);   // the adds that used the table have finished: every add waits for its stream
    cudaFree(c->counts);
    cudaFree(c->dir);
    cudaFreeHost(c->h_sizes);
    delete c;
}

int ktb_counter_add(ktb_counter *c, const uint8_t *bases, const uint64_t *offsets, uint64_t n) {
    if (!c || !offsets) return ktb_internal_fail(KTB_ERR_ARG, "counter / offsets is NULL");
    if (int rc = check_offsets(bases, offsets, n, c->k, false)) return rc;
    if (n == 0 || offsets[n] == offsets[0]) return KTB_OK;
    ktb::DeviceGuard device_guard(c->device);
    CUP(device_guard.err);

    const ChunkPlan plan(bases, offsets, n);
    // Two slots: chunk c + 1 is copied in on one stream while chunk c is counted and merged on the other.
    ChunkSlot slot[2];
    int rc = KTB_OK;
    FirstError step{rc};
    for (ChunkSlot &s : slot) s.alloc(plan, step);
    const uint64_t nchunks = plan.chunks();
    // Over several chunks, the table the add started from is kept until the add returns, so that a chunk that fails
    // (a scratch that does not fit) can restore it: the counter then holds none of the batch, not part of it.
    const ktb_counter saved = *c;
    const bool keep = nchunks > 1;
    if (rc == KTB_OK) slot[0].copy_in(plan, 0, step);
    for (uint64_t ci = 0; ci < nchunks && rc == KTB_OK; ++ci) {
        ChunkSlot &s = slot[ci & 1];
        const Chunk ch = plan[ci];
        const bool work = ch.nb > 0;
        if (work) rc = enqueue_add(c, s.bases, s.offsets, ch.n, ch.nb, s.st, !(keep && c->keys == saved.keys));
        if (rc == KTB_OK && ci + 1 < nchunks) {   // the other slot's stream finished its chunk in the last iteration
            slot[(ci + 1) & 1].copy_in(plan, ci + 1, step);
        }
        if (rc == KTB_OK && work) rc = finish_add(c, s.st);
    }
    for (ChunkSlot &s : slot) s.release(step);
    if (keep && c->keys != saved.keys) {   // the streams are idle: nothing reads either table any more
        if (rc == KTB_OK) {
            cudaFree(saved.keys);
            cudaFree(saved.counts);
        } else {
            cudaFree(c->keys);
            cudaFree(c->counts);
            c->keys = saved.keys;
            c->counts = saved.counts;
            c->nkeys = saved.nkeys;
            c->nwindows = saved.nwindows;
        }
    }
    return rc;
}

int ktb_counter_add_device(ktb_counter *c, const uint8_t *d_bases, const uint64_t *d_offsets, uint64_t n,
                           uint64_t total_bases, void *stream) {
    if (!c || !d_offsets) return ktb_internal_fail(KTB_ERR_ARG, "counter / d_offsets is NULL");
    if (total_bases > 0 && !d_bases) return ktb_internal_fail(KTB_ERR_ARG, "d_bases is NULL");
    if (n == 0 || total_bases == 0) return KTB_OK;
    ktb::DeviceGuard device_guard(c->device);
    CUP(device_guard.err);
    cudaStream_t st = (cudaStream_t)stream;
    if (int rc = enqueue_add(c, d_bases, d_offsets, n, total_bases, st)) {
        cudaStreamSynchronize(st);
        return rc;
    }
    return finish_add(c, st);
}

int ktb_counter_size(ktb_counter *c, uint64_t *nkeys, uint64_t *nwindows) {
    if (!c) return ktb_internal_fail(KTB_ERR_ARG, "counter is NULL");
    if (nkeys) *nkeys = c->nkeys;
    if (nwindows) *nwindows = c->nwindows;
    return KTB_OK;
}

int ktb_counter_read(ktb_counter *c, uint64_t *keys, uint64_t *counts, uint64_t cap) {
    if (!c) return ktb_internal_fail(KTB_ERR_ARG, "counter is NULL");
    const uint64_t m = std::min(c->nkeys, cap);
    if (m == 0 || (!keys && !counts)) return KTB_OK;
    ktb::DeviceGuard device_guard(c->device);
    CUP(device_guard.err);
    if (keys) CUP(cudaMemcpy(keys, c->keys, m * sizeof(uint64_t), cudaMemcpyDeviceToHost));
    if (counts) CUP(cudaMemcpy(counts, c->counts, m * sizeof(uint64_t), cudaMemcpyDeviceToHost));
    return KTB_OK;
}

int ktb_counter_read_device(ktb_counter *c, uint64_t *d_keys, uint64_t *d_counts, uint64_t cap, void *stream) {
    if (!c) return ktb_internal_fail(KTB_ERR_ARG, "counter is NULL");
    const uint64_t m = std::min(c->nkeys, cap);
    if (m == 0 || (!d_keys && !d_counts)) return KTB_OK;
    ktb::DeviceGuard device_guard(c->device);
    CUP(device_guard.err);
    cudaStream_t st = (cudaStream_t)stream;
    if (d_keys) CUP(cudaMemcpyAsync(d_keys, c->keys, m * sizeof(uint64_t), cudaMemcpyDeviceToDevice, st));
    if (d_counts) CUP(cudaMemcpyAsync(d_counts, c->counts, m * sizeof(uint64_t), cudaMemcpyDeviceToDevice, st));
    return KTB_OK;
}

int ktb_counter_coverage_device(ktb_counter *c, const uint8_t *d_bases, const uint64_t *d_offsets, uint64_t n,
                                uint64_t total_bases, uint32_t bin_size, uint32_t bin_count, int norm_mode,
                                int out_dtype, void *d_out, uint64_t *d_totals, void *stream) {
    if (!c || !d_offsets || (n > 0 && !d_out)) return ktb_internal_fail(KTB_ERR_ARG, "counter / d_offsets / d_out is NULL");
    if (int rc = check_coverage_args(bin_size, bin_count, norm_mode, out_dtype)) return rc;
    if (total_bases > 0 && !d_bases) return ktb_internal_fail(KTB_ERR_ARG, "d_bases is NULL");
    if (n == 0) return KTB_OK;
    ktb::DeviceGuard device_guard(c->device);
    CUP(device_guard.err);
    cudaStream_t st = (cudaStream_t)stream;
    if (int rc = ensure_dir(c, st)) return rc;
    return enqueue_coverage(c, d_bases, d_offsets, n, total_bases, bin_size, bin_count, norm_mode, out_dtype, d_out,
                            d_totals, st);
}

int ktb_counter_coverage(ktb_counter *c, const uint8_t *bases, const uint64_t *offsets, uint64_t n, uint32_t bin_size,
                         uint32_t bin_count, int norm_mode, int out_dtype, void *out, uint64_t *totals) {
    if (!c || !offsets || (n > 0 && !out)) return ktb_internal_fail(KTB_ERR_ARG, "counter / offsets / out is NULL");
    if (int rc = check_coverage_args(bin_size, bin_count, norm_mode, out_dtype)) return rc;
    if (int rc = check_offsets(bases, offsets, n, c->k, true)) return rc;
    if (n == 0) return KTB_OK;
    ktb::DeviceGuard device_guard(c->device);
    CUP(device_guard.err);

    const ChunkPlan plan(bases, offsets, n);
    const size_t esize = out_dtype == KTB_OUT_F64 ? 8 : 4;
    const uint64_t row_bytes = (uint64_t)bin_count * esize;
    // Two slots: chunk c + 1 is copied in and computed on one stream while the rows of chunk c are copied out on the
    // other.  A slot's host offsets are rewritten only after its stream has finished the chunk before.
    struct Slot : ChunkSlot {
        uint64_t *totals = nullptr;
        void *out = nullptr;
    } slot[2];
    int rc = KTB_OK;
    FirstError step{rc};
    for (Slot &s : slot) {
        s.alloc(plan, step);
        step(cudaMalloc((void **)&s.totals, plan.max_n * sizeof(uint64_t)), "cudaMalloc(totals)");
        step(cudaMalloc(&s.out, plan.max_n * row_bytes), "cudaMalloc(rows)");
    }
    if (rc == KTB_OK) rc = ensure_dir(c, slot[0].st);
    const uint64_t nchunks = plan.chunks();
    for (uint64_t ci = 0; ci < nchunks && rc == KTB_OK; ++ci) {
        Slot &s = slot[ci & 1];
        step(cudaStreamSynchronize(s.st), "cudaStreamSynchronize");   // chunk ci - 2 has left the slot
        if (rc != KTB_OK) break;
        const Chunk ch = plan[ci];
        s.copy_in(plan, ci, step);
        if (rc == KTB_OK)
            rc = enqueue_coverage(c, s.bases, s.offsets, ch.n, ch.nb, bin_size, bin_count, norm_mode, out_dtype, s.out,
                                  s.totals, s.st);
        step(cudaMemcpyAsync((char *)out + ch.i0 * row_bytes, s.out, ch.n * row_bytes, cudaMemcpyDeviceToHost, s.st),
             "cudaMemcpyAsync(rows)");
        if (totals)
            step(cudaMemcpyAsync(totals + ch.i0, s.totals, ch.n * sizeof(uint64_t), cudaMemcpyDeviceToHost, s.st),
                 "cudaMemcpyAsync(totals)");
    }
    for (Slot &s : slot) {
        s.release(step);
        cudaFree(s.totals);
        cudaFree(s.out);
    }
    return rc;
}

}  // extern "C"

// The argument checks of the coverage entry points, for the file driver's checks before any device work (file_api.cu).
__attribute__((visibility("hidden"))) int ktb_internal_coverage_args(uint32_t bin_size, uint32_t bin_count,
                                                                      int norm_mode, int out_dtype) {
    return check_coverage_args(bin_size, bin_count, norm_mode, out_dtype);
}

// The table in place, for the file driver's read-back in slices (file_api.cu).
__attribute__((visibility("hidden"))) void ktb_internal_counter_table(const ktb_counter *c, const uint64_t **keys,
                                                                       const uint64_t **counts) {
    *keys = c->keys;
    *counts = c->counts;
}
