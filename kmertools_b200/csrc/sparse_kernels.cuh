// sparse_kernels.cuh — per-sequence k-mer counts as CSR rows (ktb_sparse_vectorise*, DESIGN.md §4.5).
//
// Same histogram as the dense rows (DESIGN.md §2), stored as the distinct keys of each sequence in ascending order
// with their counts, for 1 <= k <= 31.  Pipeline of one call:
//   sparse_tile_kernel   : the base stream is cut into flat tiles of SP_T window-end positions.  A tile stages its bases
//                          (plus SP_LOOK look-back bytes of the same sequence) in shared memory, computes every window's
//                          key, radix-sorts the (piece, key) pairs in shared memory over only the 2k key bits and the
//                          piece bits (a piece = the part of one sequence inside the tile), run-length encodes them and
//                          writes the runs to the tile's slot of the pool.  Sequences inside one tile are finished here.
//   sparse_merge_kernel  : a sequence with pieces in m >= 2 tiles is merged pairwise in ceil(log2 m) rounds, one launch
//                          per round, between the two halves of the pool.  Every element finds its output position by a
//                          binary search in the partner run list; a key present in both halves keeps the summed count
//                          at its first occurrence and leaves a zero-count hole behind, so sizes never change and no
//                          round needs a scan.  The merged list of a group always starts where its first piece starts,
//                          inside the sequence's own tiles, so no sequence ever overwrites another.
//   row pointers         : exclusive u64 scans of the per-sequence distinct-key counts (row_ptr) and list lengths.
//   sparse_count_kernel / sparse_write_kernel : the lists of all sequences, holes included, laid end to end, are cut
//                          into blocks of SP_WB entries; a count pass, a scan of the block counts and a write pass drop the
//                          holes and write codes and values (normalised with make_out, values.cuh) below `cap`.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "sparse_common.cuh"
#include "values.cuh"

namespace ktb {

constexpr int SP_T = 4096;                          // window-end positions per tile
constexpr int SP_THREADS = 512;
constexpr int SP_ITEMS = SP_T / SP_THREADS;         // consecutive positions per thread
constexpr int SP_BUCKETS = 16;                      // 4-bit radix digits
constexpr uint64_t SP_NONE = ~0ull;
constexpr int SP_HEAD = 0, SP_START = 1;            // roles of a tile in a multi-tile sequence (see SparseDesc)


// shared memory of sparse_tile_kernel
constexpr size_t SP_SM_KEYS = 0;                                    // uint64_t [2][SP_T]   sort double buffer
constexpr size_t SP_SM_PC = SP_SM_KEYS + 2ull * SP_T * 8;           // uint16_t [2][SP_T]   piece of each key
constexpr size_t SP_SM_PPOS = SP_SM_PC + 2ull * SP_T * 2;           // uint16_t [SP_T + 8]  first position of each piece
constexpr size_t SP_SM_U = SP_SM_PPOS + (SP_T + 8) * 2;             // union: staged codes + start flags | digit counters |
constexpr size_t SP_SM_USIZE = 2ull * (SP_T + 8) * 2;               //        first / end run of each piece
constexpr size_t SP_SM_TOTAL = SP_SM_U + SP_SM_USIZE;
static_assert(SP_SM_USIZE >= (size_t)SP_BUCKETS * SP_THREADS * 2, "digit counters");
static_assert(SP_SM_USIZE >= (size_t)2 * SP_T + SP_LOOK, "staged codes and flags");
static_assert(SP_SM_U % 16 == 0, "alignment");

// Per tile.  Role HEAD: the tile's first piece belongs to sequence head_seq, which started in an earlier tile (tiles
// head_a..head_b).  Role START: the tile's last piece belongs to tail_seq, which starts in this tile and ends in tile
// tail_b > this one; its runs begin at tail_start in the tile's slot.  SP_NONE where a role is absent.
struct SparseDesc {
    uint64_t head_a, head_b, head_seq, tail_b, tail_seq;
    uint32_t tail_start, pad;
};

struct SparseParams {
    const uint8_t *bases;
    const uint64_t *offsets;   // n + 1, absolute
    uint64_t n;
    uint64_t ntiles;           // grid bound: ceil(total_bases / SP_T)
    uint64_t pool;             // entries per pool half (ntiles * SP_T)
    uint64_t *pkey;            // 2 * pool
    uint32_t *pcnt;            // 2 * pool
    unsigned long long *tot;   // n: valid windows                  (zeroed)
    unsigned long long *len;   // n: entries of the list, holes too (zeroed)
    unsigned long long *nnz;   // n: distinct keys                   (zeroed)
    uint64_t *loc;             // n: pool index of the final list
    SparseDesc *desc;          // ntiles (0xFF-filled)
    uint64_t *gsize;           // [2 round parities][2 roles][ntiles]: entries of the merge group starting at a tile
    uint32_t k;
    int canonical;
};

struct SparseOutParams {
    const uint64_t *V;                 // n + 1: exclusive scan of len (V[n] = entries of all lists)
    const uint64_t *loc;
    const unsigned long long *tot;
    const uint64_t *pkey;
    const uint32_t *pcnt;
    uint64_t n;
    uint64_t nblocks;                  // blocks of SP_WB entries the grid walks (bound from total_bases)
    unsigned long long *block_nnz;     // nblocks
    const unsigned long long *block_base;  // nblocks + 1 (write pass)
    uint64_t *codes;
    void *values;
    uint64_t cap;
    int norm_mode;
    int canonical;
};

// merge rounds of a sequence with pieces in m tiles: ceil(log2 m)
__host__ __device__ __forceinline__ uint32_t sp_rounds(uint64_t m) {
    uint32_t r = 0;
    while ((1ull << r) < m) ++r;
    return r;
}

// 4-bit digit at bit b of the sort key (piece << kb) | key
__device__ __forceinline__ uint32_t sp_digit(uint64_t key, uint32_t piece, uint32_t b, uint32_t kb) {
    const uint64_t lo = b < 64 ? key >> b : 0ull;
    uint32_t hi;
    if (b <= kb) hi = (kb - b) < 16 ? piece << (kb - b) : 0u;
    else hi = piece >> (b - kb);
    return (uint32_t)(lo | hi) & (SP_BUCKETS - 1);
}

// ================================================================================================
// sparse_tile_kernel — one CTA per tile of SP_T positions
// ================================================================================================
__global__ void __launch_bounds__(SP_THREADS, 2) sparse_tile_kernel(const SparseParams p) {
    extern __shared__ __align__(16) uint8_t sm[];
    uint64_t *keys = reinterpret_cast<uint64_t *>(sm + SP_SM_KEYS);
    uint16_t *pcs = reinterpret_cast<uint16_t *>(sm + SP_SM_PC);
    uint16_t *ppos = reinterpret_cast<uint16_t *>(sm + SP_SM_PPOS);
    uint8_t *codes = sm + SP_SM_U;                 // [SP_LOOK + SP_T] decoded bases of [ts - SP_LOOK, ts + SP_T)
    uint8_t *flags = codes + SP_LOOK + SP_T;       // [SP_T] 1 where a sequence starts
    uint16_t *cnt = reinterpret_cast<uint16_t *>(sm + SP_SM_U);       // [SP_BUCKETS][SP_THREADS]
    uint16_t *prb = reinterpret_cast<uint16_t *>(sm + SP_SM_U);       // [SP_T + 8] first run of each piece
    uint16_t *pre = prb + SP_T + 8;                                   // [SP_T + 8] end run of each piece
    __shared__ unsigned long long s_scan[SP_THREADS / 32];
    __shared__ uint64_t s_s0, s_s1;

    const int tid = threadIdx.x;
    const uint64_t base0 = p.offsets[0], end = p.offsets[p.n];
    const uint64_t t = blockIdx.x;
    const uint64_t ts = base0 + t * SP_T;
    if (ts >= end) return;
    const uint64_t te = min(ts + (uint64_t)SP_T, end);
    if (tid == 0) {
        s_s0 = sp_find(p.offsets, 0, p.n, ts);
        s_s1 = sp_find(p.offsets, s_s0, p.n, te - 1);
    }
    for (int i = tid; i < SP_T; i += SP_THREADS) flags[i] = 0;
    __syncthreads();
    const uint64_t s0 = s_s0, s1 = s_s1;
    const uint64_t s0start = p.offsets[s0];
    for (int i = tid; i < SP_LOOK + SP_T; i += SP_THREADS) {
        uint32_t c = 4u;
        if (ts + i >= s0start + SP_LOOK && ts + i < te + SP_LOOK) c = nt4_code(p.bases[ts + i - SP_LOOK]);
        codes[i] = (uint8_t)c;
    }
    for (uint64_t s = s0 + 1 + tid; s <= s1; s += SP_THREADS) flags[p.offsets[s] - ts] = 1;  // empty ones share a byte
    __syncthreads();

    // piece of each own position: 0 for s0, then one more at every sequence start
    const int i0 = tid * SP_ITEMS;
    unsigned long long nflag = 0, total;
#pragma unroll
    for (int j = 0; j < SP_ITEMS; ++j) nflag += flags[i0 + j];
    uint32_t pi = (uint32_t)sp_block_scan<SP_THREADS>(nflag, s_scan, total);
    const uint32_t np = 1u + (uint32_t)total;
    uint32_t piece[SP_ITEMS];
#pragma unroll
    for (int j = 0; j < SP_ITEMS; ++j) {
        if (flags[i0 + j]) ppos[++pi] = (uint16_t)(i0 + j);
        piece[j] = pi;
    }

    // keys: the reference's rolling update restarted k - 1 positions back (DESIGN.md §2)
    const uint32_t k = p.k;
    const uint64_t mask = (1ull << (2 * k)) - 1ull;
    const uint32_t shift = 2 * (k - 1);
    uint64_t f = 0, r = 0;
    uint32_t run = 0;
    for (int q = i0 - (int)(k - 1); q < i0; ++q) {
        const uint32_t c = codes[q + SP_LOOK];
        if (q >= 0 && flags[q]) run = 0;
        if (c < 4u) {
            f = ((f << 2) | c) & mask;
            r = (r >> 2) | ((uint64_t)(c ^ 3u) << shift);
            ++run;
        } else {
            run = 0;
        }
    }
    unsigned long long nvalid_mine = 0;
#pragma unroll
    for (int j = 0; j < SP_ITEMS; ++j) {
        const int q = i0 + j;
        const uint32_t c = codes[q + SP_LOOK];
        if (flags[q]) run = 0;
        if (c < 4u) {
            f = ((f << 2) | c) & mask;
            r = (r >> 2) | ((uint64_t)(c ^ 3u) << shift);
            ++run;
        } else {
            run = 0;
        }
        const bool ok = run >= k;
        keys[q] = ok ? (p.canonical ? min(f, r) : f) : 0ull;
        pcs[q] = (uint16_t)(ok ? piece[j] : np);   // np sorts invalid positions last
        nvalid_mine += ok;
    }
    unsigned long long nvalid_ull;
    sp_block_scan<SP_THREADS>(nvalid_mine, s_scan, nvalid_ull);   // also orders the staging area before its reuse
    const uint32_t nvalid = (uint32_t)nvalid_ull;

    // LSD radix sort of (piece, key) over 2k + bits(np) bits, 4 bits a pass; blocked arrangement keeps it stable
    const uint32_t kb = 2 * k;
    const uint32_t nbits = kb + (32u - __clz(np));
    int cur = 0;
    for (uint32_t b = 0; b < nbits; b += 4) {
        const uint64_t *ik = keys + cur * SP_T;
        const uint16_t *ip = pcs + cur * SP_T;
        uint64_t kk[SP_ITEMS];
        uint32_t pd[SP_ITEMS];   // piece << 4 | digit
#pragma unroll
        for (int d = 0; d < SP_BUCKETS; ++d) cnt[d * SP_THREADS + tid] = 0;
#pragma unroll
        for (int j = 0; j < SP_ITEMS; ++j) {
            kk[j] = ik[i0 + j];
            const uint32_t pc = ip[i0 + j], dg = sp_digit(kk[j], pc, b, kb);
            pd[j] = pc << 4 | dg;
            ++cnt[dg * SP_THREADS + tid];
        }
        __syncthreads();
        uint16_t *row = cnt + tid * SP_BUCKETS;   // raking scan over the counters in (digit, thread) order
        unsigned long long sum = 0;
#pragma unroll
        for (int e = 0; e < SP_BUCKETS; ++e) sum += row[e];
        uint32_t acc = (uint32_t)sp_block_scan<SP_THREADS>(sum, s_scan, total);
#pragma unroll
        for (int e = 0; e < SP_BUCKETS; ++e) {
            const uint32_t v = row[e];
            row[e] = (uint16_t)acc;
            acc += v;
        }
        __syncthreads();
        uint64_t *ok_ = keys + (cur ^ 1) * SP_T;
        uint16_t *op = pcs + (cur ^ 1) * SP_T;
#pragma unroll
        for (int j = 0; j < SP_ITEMS; ++j) {
            const uint32_t pos = cnt[(pd[j] & (SP_BUCKETS - 1)) * SP_THREADS + tid]++;
            ok_[pos] = kk[j];
            op[pos] = (uint16_t)(pd[j] >> 4);
        }
        __syncthreads();
        cur ^= 1;
    }

    // run-length encoding of the sorted valid pairs
    const uint64_t *sk = keys + cur * SP_T;
    const uint16_t *sp = pcs + cur * SP_T;
    uint32_t *rstart = reinterpret_cast<uint32_t *>(keys + (cur ^ 1) * SP_T);   // [SP_T + 1] first item of each run
    for (uint32_t i = tid; i <= np; i += SP_THREADS) prb[i] = pre[i] = 0;
    bool hd[SP_ITEMS];
    unsigned long long nhead = 0;
#pragma unroll
    for (int j = 0; j < SP_ITEMS; ++j) {
        const uint32_t i = i0 + j;
        hd[j] = i < nvalid && (i == 0 || sk[i] != sk[i - 1] || sp[i] != sp[i - 1]);
        nhead += hd[j];
    }
    unsigned long long nruns_ull;
    uint32_t ridx = (uint32_t)sp_block_scan<SP_THREADS>(nhead, s_scan, nruns_ull);   // also orders prb / pre zeroing
    const uint32_t nruns = (uint32_t)nruns_ull;
#pragma unroll
    for (int j = 0; j < SP_ITEMS; ++j) {
        const uint32_t i = i0 + j;
        if (i < nvalid) {
            if (hd[j]) rstart[ridx++] = i;
            if (i == 0 || sp[i] != sp[i - 1]) prb[sp[i]] = (uint16_t)(ridx - 1);
            if (i == nvalid - 1 || sp[i + 1] != sp[i]) pre[sp[i]] = (uint16_t)ridx;
        }
    }
    if (tid == 0) rstart[nruns] = nvalid;
    __syncthreads();

    const uint64_t slot = t * SP_T;
    for (uint32_t q = tid; q < nruns; q += SP_THREADS) {
        const uint32_t i = rstart[q];
        p.pkey[slot + q] = sk[i];
        p.pcnt[slot + q] = rstart[q + 1] - i;
    }
    for (uint32_t q = tid; q < np; q += SP_THREADS) {
        const uint64_t s = q == 0 ? s0 : sp_find(p.offsets, s0, s1 + 1, ts + ppos[q]);
        const uint64_t start = p.offsets[s], stop = p.offsets[s + 1];
        const uint32_t rb = prb[q], runs = pre[q] - rb;
        const uint32_t windows = runs ? rstart[rb + runs] - rstart[rb] : 0u;
        if (start >= ts && stop <= te) {   // the whole sequence is in this tile: its row is final
            p.tot[s] = windows;
            p.len[s] = runs;
            p.nnz[s] = runs;
            p.loc[s] = slot + rb;
            continue;
        }
        if (runs) {
            atomicAdd(p.tot + s, (unsigned long long)windows);
            atomicAdd(p.len + s, (unsigned long long)runs);
            atomicAdd(p.nnz + s, (unsigned long long)runs);
        }
        if (start >= ts) {   // starts here, continues: the last piece; its merged list will start where its runs start
            const uint64_t b = (stop - 1 - base0) / SP_T;
            const uint32_t tail_start = nruns - runs;
            p.loc[s] = ((sp_rounds(b - t + 1) & 1u) ? p.pool : 0ull) + slot + tail_start;
            p.desc[t].tail_b = b;
            p.desc[t].tail_seq = s;
            p.desc[t].tail_start = tail_start;
            p.gsize[(uint64_t)SP_START * p.ntiles + t] = runs;
        } else {             // piece 0 of a sequence that started in an earlier tile
            p.desc[t].head_a = (start - base0) / SP_T;
            p.desc[t].head_b = (stop - 1 - base0) / SP_T;
            p.desc[t].head_seq = s;
            p.gsize[(uint64_t)SP_HEAD * p.ntiles + t] = runs;
        }
    }
}

// ================================================================================================
// sparse_merge_kernel — round r (1-based) of the pairwise merge; one CTA walks the pool slot of one tile at a time
// ================================================================================================
__global__ void __launch_bounds__(SP_MTHREADS) sparse_merge_kernel(const SparseParams p, uint32_t r) {
    __shared__ unsigned long long s_scan[SP_MTHREADS / 32];
    const uint32_t sh = r - 1;
    const uint64_t h = 1ull << sh;
    const uint64_t src = (sh & 1u) ? p.pool : 0ull, dst = (r & 1u) ? p.pool : 0ull;
    const uint64_t *skey = p.pkey + src;
    const uint32_t *scnt = p.pcnt + src;
    uint64_t *dkey = p.pkey + dst;
    uint32_t *dcnt = p.pcnt + dst;
    const uint64_t *gin = p.gsize + (uint64_t)(sh & 1u) * 2 * p.ntiles;
    uint64_t *gout = p.gsize + (uint64_t)(r & 1u) * 2 * p.ntiles;
    for (uint64_t x = blockIdx.x; x < p.ntiles; x += gridDim.x) {
        const SparseDesc d = p.desc[x];
        for (int role = SP_HEAD; role <= SP_START; ++role) {
            uint64_t a, b, s;
            if (role == SP_HEAD) {
                if (d.head_a == SP_NONE) continue;
                a = d.head_a; b = d.head_b; s = d.head_seq;
            } else {
                if (d.tail_b == SP_NONE) continue;
                a = x; b = d.tail_b; s = d.tail_seq;
            }
            if (r > sp_rounds(b - a + 1)) continue;   // this sequence is finished
            const uint64_t off_a = role == SP_START ? d.tail_start : p.desc[a].tail_start;
            // group g of round r - 1 holds tile x; it merges with its neighbour g ^ 1
            const uint64_t g = (x - a) >> sh;
            const uint64_t xg = a + (g << sh);
            const uint64_t start_g = xg * SP_T + (xg == a ? off_a : 0);
            const uint64_t size_g = gin[(uint64_t)(xg == a ? SP_START : SP_HEAD) * p.ntiles + xg];
            const bool left = (g & 1) == 0;
            const uint64_t xp = left ? xg + h : xg - h;
            const bool has = !left || xp <= b;
            const uint64_t start_p = has ? xp * SP_T + (xp == a ? off_a : 0) : 0;
            const uint64_t size_p = has ? gin[(uint64_t)(xp == a ? SP_START : SP_HEAD) * p.ntiles + xp] : 0;
            if (left && x == xg && threadIdx.x == 0) gout[(uint64_t)(xg == a ? SP_START : SP_HEAD) * p.ntiles + xg] = size_g + size_p;
            const uint64_t lo = max(start_g, x * SP_T), hi = min(start_g + size_g, x * SP_T + SP_T);
            unsigned long long absorbed = 0;
            for (uint64_t q = lo + threadIdx.x; q < hi; q += SP_MTHREADS) {
                const uint64_t key = skey[q];
                uint32_t c = scnt[q];
                const uint64_t j = q - start_g;
                uint64_t pos;
                if (left) {   // ties: the left list first; a key's first occurrence carries its whole count
                    const uint64_t lb = sp_lower_bound(skey + start_p, size_p, key);
                    if (c && lb < size_p && skey[start_p + lb] == key) c += scnt[start_p + lb];
                    pos = start_g + j + lb;
                } else {
                    const uint64_t ub = sp_upper_bound(skey + start_p, size_p, key);
                    if (ub && skey[start_p + ub - 1] == key) {
                        absorbed += c != 0;
                        c = 0;
                    }
                    pos = start_p + j + ub;
                }
                dkey[pos] = key;
                dcnt[pos] = c;
            }
            unsigned long long total;
            sp_block_scan<SP_MTHREADS>(absorbed, s_scan, total);
            if (threadIdx.x == 0 && total) atomicAdd(p.nnz + s, 0ull - total);
        }
    }
}

// ================================================================================================
// write-out: the lists of all sequences end to end (V), blocks of SP_WB entries, holes dropped
// ================================================================================================
template <typename F>
__device__ __forceinline__ void sp_walk(const SparseOutParams &o, uint64_t v0, uint64_t v1, uint64_t slo, uint64_t shi,
                                        F fn) {
    const uint64_t a = v0 + (uint64_t)threadIdx.x * SP_WITEMS;
    const uint64_t e = min(a + SP_WITEMS, v1);
    if (a >= e) return;
    uint64_t s = sp_find(o.V, slo, shi + 1, a);
    for (uint64_t v = a; v < e; ++v) {
        while (o.V[s + 1] <= v) ++s;
        const uint64_t q = o.loc[s] + (v - o.V[s]);
        fn(s, q, o.pcnt[q]);
    }
}

// entries [v0, v1) of block blk and the sequences [slo, shi] they belong to; false past the last entry
__device__ __forceinline__ bool sp_block_range(const SparseOutParams &o, uint64_t blk, uint64_t &v0, uint64_t &v1,
                                               uint64_t &slo, uint64_t &shi, uint64_t *s_range) {
    const uint64_t vtot = o.V[o.n];
    v0 = blk * SP_WB;
    if (v0 >= vtot) return false;
    v1 = min(v0 + SP_WB, vtot);
    if (threadIdx.x == 0) {
        s_range[0] = sp_find(o.V, 0, o.n, v0);
        s_range[1] = sp_find(o.V, s_range[0], o.n, v1 - 1);
    }
    __syncthreads();
    slo = s_range[0];   // read before the block scan that follows, so thread 0 cannot overwrite it early
    shi = s_range[1];
    return true;
}

__global__ void __launch_bounds__(SP_MTHREADS) sparse_count_kernel(const SparseOutParams o) {
    __shared__ unsigned long long s_scan[SP_MTHREADS / 32];
    __shared__ uint64_t s_range[2];
    for (uint64_t blk = blockIdx.x; blk < o.nblocks; blk += gridDim.x) {
        uint64_t v0, v1, slo, shi;
        if (!sp_block_range(o, blk, v0, v1, slo, shi, s_range)) {
            if (threadIdx.x == 0) o.block_nnz[blk] = 0;
            continue;
        }
        unsigned long long mine = 0, total;
        sp_walk(o, v0, v1, slo, shi, [&](uint64_t, uint64_t, uint32_t c) { mine += c != 0; });
        sp_block_scan<SP_MTHREADS>(mine, s_scan, total);
        if (threadIdx.x == 0) o.block_nnz[blk] = total;
    }
}

template <int OUT>
__global__ void __launch_bounds__(SP_MTHREADS) sparse_write_kernel(const SparseOutParams o) {
    using T = typename OutT<OUT>::type;
    T *values = reinterpret_cast<T *>(o.values);
    const bool norm = o.norm_mode != NORM_COUNTS;
    __shared__ unsigned long long s_scan[SP_MTHREADS / 32];
    __shared__ uint64_t s_range[2];
    for (uint64_t blk = blockIdx.x; blk < o.nblocks; blk += gridDim.x) {
        uint64_t v0, v1, slo, shi;
        if (!sp_block_range(o, blk, v0, v1, slo, shi, s_range)) continue;
        unsigned long long mine = 0, total;
        sp_walk(o, v0, v1, slo, shi, [&](uint64_t, uint64_t, uint32_t c) { mine += c != 0; });
        uint64_t at = o.block_base[blk] + sp_block_scan<SP_MTHREADS>(mine, s_scan, total);
        if (mine == 0 || at >= o.cap) continue;
        sp_walk(o, v0, v1, slo, shi, [&](uint64_t s, uint64_t q, uint32_t c) {
            if (c == 0) return;
            if (at < o.cap) {
                const uint64_t dv = norm_divisor(o.tot[s], o.norm_mode, o.canonical);
                const float dF = (float)dv;
                o.codes[at] = o.pkey[q];
                values[at] = make_out<OUT>(c, norm, dv < (1ull << 24), dF, __frcp_rn(dF), (double)dv);
            }
            ++at;
        });
    }
}

// ================================================================================================
// exclusive u64 scan: out[0..n] (out[n] = sum), three launches (block sums, one-CTA scan of those, block scans)
// ================================================================================================
__device__ __forceinline__ unsigned long long sp_thread_sum(const unsigned long long *in, uint64_t n, uint64_t i0) {
    unsigned long long s = 0;
#pragma unroll
    for (int j = 0; j < SP_WITEMS; ++j)
        if (i0 + j < n) s += in[i0 + j];
    return s;
}

__global__ void __launch_bounds__(SP_MTHREADS) sparse_scan_reduce_kernel(const unsigned long long *in, uint64_t n,
                                                                         unsigned long long *bsum) {
    __shared__ unsigned long long s_scan[SP_MTHREADS / 32];
    const uint64_t i0 = (uint64_t)blockIdx.x * SP_WB + (uint64_t)threadIdx.x * SP_WITEMS;
    unsigned long long total;
    sp_block_scan<SP_MTHREADS>(sp_thread_sum(in, n, i0), s_scan, total);
    if (threadIdx.x == 0) bsum[blockIdx.x] = total;
}

__global__ void __launch_bounds__(1024) sparse_scan_top_kernel(unsigned long long *bsum, uint64_t nb,
                                                               unsigned long long *out_total) {
    __shared__ unsigned long long s_scan[32];
    unsigned long long carry = 0;
    for (uint64_t b0 = 0; b0 < nb; b0 += 1024) {
        const uint64_t b = b0 + threadIdx.x;
        const unsigned long long v = b < nb ? bsum[b] : 0ull;
        unsigned long long total;
        const unsigned long long ex = sp_block_scan<1024>(v, s_scan, total);
        if (b < nb) bsum[b] = carry + ex;
        carry += total;
    }
    if (threadIdx.x == 0) *out_total = carry;
}

__global__ void __launch_bounds__(SP_MTHREADS) sparse_scan_down_kernel(const unsigned long long *in, uint64_t n,
                                                                       const unsigned long long *bsum,
                                                                       unsigned long long *out) {
    __shared__ unsigned long long s_scan[SP_MTHREADS / 32];
    const uint64_t i0 = (uint64_t)blockIdx.x * SP_WB + (uint64_t)threadIdx.x * SP_WITEMS;
    unsigned long long total;
    unsigned long long acc = bsum[blockIdx.x] + sp_block_scan<SP_MTHREADS>(sp_thread_sum(in, n, i0), s_scan, total);
#pragma unroll
    for (int j = 0; j < SP_WITEMS; ++j)
        if (i0 + j < n) {
            const unsigned long long v = in[i0 + j];
            out[i0 + j] = acc;
            acc += v;
        }
}

}  // namespace ktb
