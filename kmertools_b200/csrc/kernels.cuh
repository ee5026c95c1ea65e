// kernels.cuh — sm_100a device code of the oligonucleotide-frequency-vector path.
//
// What is computed (closed form of kmer/src/kmer.rs:80-106 + composition/src/oligo.rs:231-259,
// see DESIGN.md §2):
//   c[p]      = nt4(seq[p])                       0..3 valid, 4 ambiguous       (kmer.rs:6-15)
//   valid(p)  = the k bases ending at p are all < 4
//   f(p)      = sum_j c[p-k+1+j] * 4^(k-1-j)       forward code, oldest base most significant
//   r(p)      = sum_j (3-c[p-k+1+j]) * 4^j         reverse complement in the same encoding
//   row[rank(min(f,r))] += 1  (canonical)   |   row[f] += 1  (raw)          for every valid p
//   row[j]   /= max(1, total)                      when normalising
//
// Kernels of this file (DESIGN.md §4; long_kernel.cuh and bucket_kernels.cuh hold the round-2 kernels):
//   short_kernel  : one WARP per group of 16 short reads (<= 255 windows each, 4^k <= 1024): read-aligned
//                   16-base chunks per lane, byte counters packed four to a word, shared-memory atomics,
//                   linear coalesced write-out with fused normalisation.  Groups it cannot take go to a
//                   reject list.
//   seq_kernel    : one CTA per sequence (consumes the reject list, or everything when k is large): warps walk
//                   contiguous runs of 32-chunk steps with a carried look-back word; histogram in shared
//                   memory in code space (mode 1), dense middle-base space (mode 4, k = 7), rank space
//                   (mode 2 / 7, k = 8), packed 16-bit rank space (mode 5), raw (mode 0), or straight
//                   into zeroed global rows with RED atomics for histograms larger than shared memory
//                   (mode 3, driven in L2-sized waves by the host).  long_kernel replaces it for k = 7 and for
//                   long sequences at k <= 5 (u32 / f32 rows).
//   wave_kernel   : rows larger than shared memory as ONE persistent cooperative launch (global RED atomics in
//                   L2-sized waves).  Round 2 replaced it by bucket_kernel + count_kernel for k <= 10; it stays
//                   the path for k = 11, 12 and behind the option bucket = 0.
//   finalize_kernel: u32 counts -> f32 / f64 rows for mode 3.
//   flat_kernel   : flat decomposition of the base stream + global atomics; cross-check only (force_path=1).
#pragma once
#include <cooperative_groups.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "values.cuh"

#ifndef KTB_SEQ_MAXTHREADS
#define KTB_SEQ_MAXTHREADS 256
#endif
#ifndef KTB_SEQ_MINBLOCKS
#define KTB_SEQ_MINBLOCKS 3
#endif
#ifndef KTB_SEQ_MINBLOCKS4
#define KTB_SEQ_MINBLOCKS4 6
#endif
#ifndef KTB_SEQ_FASTPATH
#define KTB_SEQ_FASTPATH 1
#endif

namespace ktb {

__global__ void nt4_table_kernel(uint8_t *out) { out[threadIdx.x] = (uint8_t)nt4_code(threadIdx.x); }

// ================================================================================================
// shared decode helpers (16 bases per lane from one 128-bit word group)
// ================================================================================================

// 16 bases -> packed 2-bit codes (base j at bits 2*(15-j)+1..2*(15-j), oldest base most significant)
// and a 16-bit validity mask (base j at bit 15-j).
__device__ __forceinline__ void decode16(const uint4 v, uint32_t &cf, uint32_t &vm) {
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
    uint32_t m[4];
    bool all_ok = true;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const uint32_t c4 = ((w[q] >> 1) ^ (w[q] >> 2)) & 0x03030303u;
        m[q] = c4 * 0x40100401u;  // top byte = b0<<6 | b1<<4 | b2<<2 | b3
        // validity: rebuild the upper-case letter each code stands for and compare with the input
        const uint32_t y = (c4 | (c4 >> 4)) & 0x00FF00FFu;
        const uint32_t sel = (y | (y >> 8)) & 0xFFFFu;
        const uint32_t recon = __byte_perm(0x54474341u, 0u, sel);  // "ACGT"[code]
        all_ok &= (recon == (w[q] & 0xDFDFDFDFu));
    }
    const uint32_t u01 = __byte_perm(m[1], m[0], 0x0073);
    const uint32_t u23 = __byte_perm(m[3], m[2], 0x0073);
    cf = __byte_perm(u23, u01, 0x5410);
    vm = 0xFFFFu;
    if (!all_ok) {  // N / IUPAC / U / raw 0..3 codes somewhere in the warp: exact path, four bytes at a time
        // zero-byte detector: bit 7 of every byte of the result is set iff that byte of x is 0
        auto zero_bytes = [](uint32_t x) { return ~(((x & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | x) & 0x80808080u; };
        vm = 0;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const uint32_t u = w[q] & 0xDFDFDFDFu;
            uint32_t c4 = ((w[q] >> 1) ^ (w[q] >> 2)) & 0x03030303u;          // right for A C G T U, either case
            const uint32_t y = (c4 | (c4 >> 4)) & 0x00FF00FFu;
            const uint32_t recon = __byte_perm(0x54474341u, 0u, (y | (y >> 8)) & 0xFFFFu);
            const uint32_t raw = zero_bytes(w[q] & 0xFCFCFCFCu);               // bytes 0..3 are their own code
            const uint32_t ok = zero_bytes(recon ^ u) | zero_bytes(u ^ 0x55555555u) | raw;
            const uint32_t rawff = (raw >> 7) * 0xFFu;
            c4 = (c4 & ~rawff) | (w[q] & 0x03030303u & rawff);
            m[q] = c4 * 0x40100401u;
            vm = (vm << 4) | ((((ok >> 7) * 0x08040201u) >> 24) & 0xFu);       // first base of the word = highest bit
        }
        const uint32_t v01 = __byte_perm(m[1], m[0], 0x0073);
        const uint32_t v23 = __byte_perm(m[3], m[2], 0x0073);
        cf = __byte_perm(v23, v01, 0x5410);
    }
}

// reverse-complement packing of 16 bases: base j at bits 2j+1..2j, complemented
__device__ __forceinline__ uint32_t revcomp_pack(uint32_t cf) {
    uint32_t x = __brev(~cf);
    return ((x >> 1) & 0x55555555u) | ((x & 0x55555555u) << 1);
}

// bit b of the result is set <=> bits b..b+k-1 of V are all set (older bases = higher bits)
__device__ __forceinline__ uint32_t window_mask(uint32_t V, uint32_t k) {
    uint32_t vw = V, have = 1;
    while (have < k) {
        const uint32_t step = min(have, k - have);
        vw &= vw >> step;
        have += step;
    }
    return vw;
}

// 16 bytes at p (16-byte aligned offset into bases) without touching memory at or beyond `total`
__device__ __forceinline__ uint4 load16_guarded(const uint8_t *bases, uint64_t p, uint64_t total) {
    if (p + 16 <= total) return __ldg(reinterpret_cast<const uint4 *>(bases + p));
    uint32_t t[4] = {0x41414141u, 0x41414141u, 0x41414141u, 0x41414141u};  // filler decodes on the fast path
    for (uint64_t b = p; b < total; ++b) {
        const uint32_t sh = (uint32_t)(b - p);
        t[sh >> 2] = (t[sh >> 2] & ~(0xFFu << ((sh & 3) * 8))) | ((uint32_t)bases[b] << ((sh & 3) * 8));
    }
    return make_uint4(t[0], t[1], t[2], t[3]);
}

// ================================================================================================
// short_kernel — one warp per group of G consecutive short reads, 16 bases per lane per step
// ================================================================================================
struct ShortParams {
    const uint8_t *bases;     // 16-byte aligned
    const uint64_t *offsets;
    uint64_t n;
    uint64_t ngroups;         // ceil(n / G)
    uint64_t total_bases;
    void *out;
    uint64_t *totals;         // optional
    const uint32_t *tab;      // [4^k] code -> (byte offset of the bin's word << 22) | (8 * (bin & 3))
    unsigned long long *counter;        // dynamic group counter (zeroed before launch)
    uint32_t *reject_list;              // groups this kernel does not take (consumed by seq_kernel)
    unsigned long long *reject_count;   // zeroed before launch
    uint32_t k;
    uint32_t ncodes;          // 4^k  (<= 1024)
    uint32_t dim;             // row width, multiple of 4
    uint32_t words;           // dim / 4 : 32-bit histogram words per read (4 byte counters each)
    uint32_t words_recip;     // ceil(2^32 / words)
    uint32_t max_len;         // longest read this kernel takes: 254 + k (<= 255 windows fit a byte)
    int norm_mode;
    int canonical;
};

constexpr int SHORT_MAX_CODES = 1024;
constexpr int SHORT_G = 16;   // reads per warp-group
constexpr int SHORT_PAD = 64;  // per-warp scratch words after the histograms (totals, divisors)

// Work decomposition: the reads of a group are cut into read-aligned 16-base chunks; chunk t of the
// group goes to lane t%32 of step t/32, so all 16 windows a lane emits belong to one read and one
// histogram.  A lane fetches its (unaligned) 16 bytes with two aligned 128-bit loads and a byte funnel,
// turns them into a 2-bit packed word + validity mask, gets the previous chunk's word from its
// neighbour lane by shuffle (look-back for windows straddling chunks) and cuts the k-mers out of the
// 64-bit window.  Counters are bytes packed four to a word (a short read has <= 255 windows), updated
// with shared-memory atomics (measured 13-15 random updates/cycle/SM, profiles/r1_microbench*.txt).
// Write-out walks the group's histograms linearly: one word -> four floats -> one 128-bit store.
template <int OUT, bool NORM>
__global__ void __launch_bounds__(256) short_kernel(const ShortParams p) {
    extern __shared__ __align__(16) uint32_t smem_u32[];
    __shared__ uint32_t s_tab[SHORT_MAX_CODES];

    constexpr int G = SHORT_G;
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    for (uint32_t i = threadIdx.x; i < p.ncodes; i += blockDim.x) s_tab[i] = p.tab[i];

    const uint32_t hwords = G * p.words;                    // histogram words per warp
    uint32_t *hist = smem_u32 + (size_t)warp * (hwords + SHORT_PAD);
    uint32_t *s_tot = hist + hwords;                        // [G] valid windows per read
    float *s_df = reinterpret_cast<float *>(s_tot + G);     // [G] divisor as float
    float *s_ri = reinterpret_cast<float *>(s_tot + 2 * G); // [G] RN(1 / divisor)
    for (uint32_t i = lane; i < hwords + SHORT_PAD; i += 32) hist[i] = 0;
    __syncthreads();

    const uint32_t k = p.k;
    const uint32_t kmask4 = ((1u << (2 * k)) - 1u) << 2;   // k-mer code pre-scaled to a byte offset into s_tab
    using T = typename OutT<OUT>::type;
    T *out = reinterpret_cast<T *>(p.out);
    constexpr uint32_t FULL = 0xffffffffu;

    for (;;) {
        unsigned long long g = 0;
        if (lane == 0) g = atomicAdd(p.counter, 1ULL);
        g = __shfl_sync(FULL, g, 0);
        if (g >= p.ngroups) break;
        const uint64_t i0 = g * (uint64_t)G;
        const uint32_t nreads = (uint32_t)min((unsigned long long)G, (unsigned long long)(p.n - i0));
        // lane j < nreads owns read i0+j
        uint64_t o0 = 0, o1 = 0;
        if ((uint32_t)lane < nreads) {
            o0 = p.offsets[i0 + lane];
            o1 = p.offsets[i0 + lane + 1];
        }
        const uint64_t lenl = o1 - o0;
        if (!__all_sync(FULL, lenl <= (uint64_t)p.max_len)) {
            if (lane == 0) p.reject_list[atomicAdd(p.reject_count, 1ULL)] = (uint32_t)g;
            continue;
        }
        const uint32_t len = (uint32_t)lenl;
        const uint64_t gbase = __shfl_sync(FULL, o0, 0);
        const uint32_t rel = (uint32_t)(o0 - gbase);        // start of my read relative to the group
        const uint32_t cnt = (len + 15u) >> 4;              // 16-base chunks in my read
        uint32_t cum = cnt;                                 // inclusive prefix sum over lanes
#pragma unroll
        for (int s = 1; s < 32; s <<= 1) {
            const uint32_t v = __shfl_up_sync(FULL, cum, s);
            if (lane >= s) cum += v;
        }
        const uint32_t ex = cum - cnt;                      // first chunk index of my read
        const uint32_t ntasks = __shfl_sync(FULL, cum, 31);
        const uint32_t len0 = __shfl_sync(FULL, len, 0);
        const bool uniform = __all_sync(FULL, (uint32_t)lane >= nreads || len == len0) && len0 > 0;
        const uint32_t cpr = (len0 + 15u) >> 4;
        const uint32_t cpr_recip = uniform ? (0xFFFFFFFFu / cpr + 1u) : 0u;

        uint32_t carry_cf = 0, carry_vm = 0;
        // one step = 32 chunk tasks; the loads of step s+1 are issued before step s is processed
        struct Task { uint32_t r, q, a, nvalid; bool active; uint4 v0, v1; };
        auto fetch_task = [&](uint32_t t0) -> Task {
            Task tk;
            const uint32_t t = t0 + lane;
            tk.active = t < ntasks;
            uint32_t r, q;
            if (uniform) {
                r = (cpr == 1) ? t : __umulhi(t, cpr_recip);
                q = t - r * cpr;
            } else {
                r = 0;
                uint32_t exr = 0;
#pragma unroll
                for (int s = 16; s > 0; s >>= 1) {  // largest r with ex[r] <= t
                    const uint32_t cand = r + s;
                    const uint32_t v = __shfl_sync(FULL, ex, cand & 31);
                    if (cand < nreads && v <= t) { r = cand; exr = v; }
                }
                q = t - exr;
            }
            r = tk.active ? r : 0;
            const uint32_t rrel = __shfl_sync(FULL, rel, r);
            const uint32_t rlen = __shfl_sync(FULL, len, r);
            tk.r = r; tk.q = q; tk.a = 0; tk.nvalid = 0;
            tk.v0 = tk.v1 = make_uint4(0x41414141u, 0x41414141u, 0x41414141u, 0x41414141u);
            if (tk.active) {
                const uint64_t addr = gbase + rrel + 16u * q;
                tk.nvalid = min(16u, rlen - 16u * q);
                tk.a = (uint32_t)addr & 15u;
                const uint64_t pa = addr - tk.a;
                tk.v0 = load16_guarded(p.bases, pa, p.total_bases);
                if (tk.a + tk.nvalid > 16u) tk.v1 = load16_guarded(p.bases, pa + 16, p.total_bases);
            }
            return tk;
        };
        Task cur = fetch_task(0);
        for (uint32_t t0 = 0; t0 < ntasks; t0 += 32) {
            Task nxt = cur;
            if (t0 + 32 < ntasks) nxt = fetch_task(t0 + 32);
            const uint32_t r = cur.r, q = cur.q;
            uint32_t cf = (uint32_t)lane * 0x9E3779B1u, vm = 0;  // idle lanes add 0 at scattered bins
            if (cur.active) {
                const uint32_t a = cur.a;
                uint4 u = cur.v0;
                if (a) {   // byte funnel: u = bytes a..a+15 of (v0 : v1)
                    const uint4 v0 = cur.v0, v1 = cur.v1;
                    uint32_t W0 = v0.x, W1 = v0.y, W2 = v0.z, W3 = v0.w, W4 = v1.x, W5 = v1.y, W6 = v1.z, W7 = v1.w;
                    if (a & 8u) { W0 = W2; W1 = W3; W2 = W4; W3 = W5; W4 = W6; W5 = W7; }
                    if (a & 4u) { W0 = W1; W1 = W2; W2 = W3; W3 = W4; W4 = W5; }
                    const uint32_t bs = (a & 3u) * 8u;
                    u.x = __funnelshift_r(W0, W1, bs);
                    u.y = __funnelshift_r(W1, W2, bs);
                    u.z = __funnelshift_r(W2, W3, bs);
                    u.w = __funnelshift_r(W3, W4, bs);
                }
                decode16(u, cf, vm);
                vm &= (0xFFFF0000u >> cur.nvalid) & 0xFFFFu;   // bases past the end of the read
            }
            cur = nxt;
            uint32_t cf_prev = __shfl_up_sync(FULL, cf, 1);
            uint32_t vm_prev = __shfl_up_sync(FULL, vm, 1);
            if (lane == 0) { cf_prev = carry_cf; vm_prev = carry_vm; }
            carry_cf = __shfl_sync(FULL, cf, 31);
            carry_vm = __shfl_sync(FULL, vm, 31);
            if (q == 0) vm_prev = 0;                       // first chunk of a read: no look-back
            const uint32_t vw = window_mask((vm_prev << 16) | vm, k) & 0xFFFFu;
            if (vw) atomicAdd(&s_tot[r], (uint32_t)__popc(vw));
            // all 16 table look-ups first (independent, pipelined), then the atomics
            const uint64_t F4 = (((uint64_t)cf_prev << 32) | cf) << 2;
            uint8_t *hb = reinterpret_cast<uint8_t *>(hist + r * p.words);
            uint32_t e[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                const uint32_t idx4 = (uint32_t)(F4 >> (2 * (15 - j))) & kmask4;
                e[j] = *reinterpret_cast<const uint32_t *>(reinterpret_cast<const uint8_t *>(s_tab) + idx4);
            }
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                // branch-free: an invalid window adds 0 (ptxas turns a predicated ATOMS into a branch)
                const uint32_t one = (vw >> (15 - j)) & 1u;
                atomicAdd(reinterpret_cast<uint32_t *>(hb + (e[j] >> 22)), one << (e[j] & 31u));
            }
        }
        __syncwarp();

        // ---- write-out: linear sweep over the group's histograms (rows are contiguous in `out`)
        if ((uint32_t)lane < nreads) {
            const uint32_t tot = s_tot[lane];
            if (p.totals) p.totals[i0 + lane] = tot;
            const float dF = (float)norm_divisor(tot, p.norm_mode, p.canonical);  // <= 510, exact
            s_df[lane] = dF;
            s_ri[lane] = __frcp_rn(dF);
        }
        __syncwarp();
        T *obase = out + i0 * (uint64_t)p.dim;
        const uint32_t nw = nreads * p.words;
        for (uint32_t i = lane; i < nw; i += 32) {
            const uint32_t r = (p.words == 1u) ? i : __umulhi(i, p.words_recip);
            const uint32_t v = hist[i];
            const float dF = s_df[r];
            const float rinv = s_ri[r];
            T e0, e1, e2, e3;
            if constexpr (OUT == OUT_U32) {
                e0 = v & 0xFFu; e1 = (v >> 8) & 0xFFu; e2 = (v >> 16) & 0xFFu; e3 = v >> 24;
            } else {
                // byte -> float without I2F: 0x4B000000 | b is the float 2^23 + b
                const float c0 = __uint_as_float(__byte_perm(v, 0x4B000000u, 0x7440)) - 8388608.0f;
                const float c1 = __uint_as_float(__byte_perm(v, 0x4B000000u, 0x7441)) - 8388608.0f;
                const float c2 = __uint_as_float(__byte_perm(v, 0x4B000000u, 0x7442)) - 8388608.0f;
                const float c3 = __uint_as_float(__byte_perm(v, 0x4B000000u, 0x7443)) - 8388608.0f;
                if constexpr (OUT == OUT_F32) {
                    e0 = NORM ? quot_f32(c0, dF, rinv) : c0;
                    e1 = NORM ? quot_f32(c1, dF, rinv) : c1;
                    e2 = NORM ? quot_f32(c2, dF, rinv) : c2;
                    e3 = NORM ? quot_f32(c3, dF, rinv) : c3;
                } else {
                    const double dD = (double)dF;
                    e0 = NORM ? (double)c0 / dD : (double)c0;
                    e1 = NORM ? (double)c1 / dD : (double)c1;
                    e2 = NORM ? (double)c2 / dD : (double)c2;
                    e3 = NORM ? (double)c3 / dD : (double)c3;
                }
            }
            T *dstp = obase + (uint64_t)i * 4u;
            if constexpr (OUT == OUT_F64) {
                reinterpret_cast<double2 *>(dstp)[0] = make_double2(e0, e1);
                reinterpret_cast<double2 *>(dstp)[1] = make_double2(e2, e3);
            } else if constexpr (OUT == OUT_F32) {
                *reinterpret_cast<float4 *>(dstp) = make_float4(e0, e1, e2, e3);
            } else {
                *reinterpret_cast<uint4 *>(dstp) = make_uint4(e0, e1, e2, e3);
            }
        }
        __syncwarp();
        {
            uint4 *hz = reinterpret_cast<uint4 *>(hist);
            for (uint32_t i = lane; i < (hwords + SHORT_PAD) / 4; i += 32) hz[i] = make_uint4(0, 0, 0, 0);
        }
        __syncwarp();
    }
}

// ================================================================================================
// seq_kernel — CTA per sequence, shared-memory atomics
// ================================================================================================
struct SeqParams {
    uint32_t grab = 1;            // consecutive work items taken per atomic on `counter`
    const uint8_t *bases;        // 16-byte aligned
    const uint64_t *offsets;
    uint64_t n;
    uint64_t total_bases;
    void *out;
    uint64_t *totals;            // optional
    const uint32_t *rank_full;   // [4^k] code -> rank of its canonical form (rank-space mode)
    const uint32_t *canon_of_rank;  // [dim] rank -> canonical code       (code-space mode)
    const uint32_t *canon_perm;     // canon_of_rank permuted inside 128-rank blocks: [b*128+4l+e] = canon[b*128+32e+l]
    unsigned long long *counter; // dynamic group counter (zeroed before launch)
    uint32_t k;
    uint32_t dim;
    uint32_t hist_entries;       // shared-memory histogram entries (4^k in code space, dim in rank space)
    int norm_mode;
    int canonical;
    const uint32_t *list;        // groups to process (short_kernel's rejects); nullptr = every group
    const unsigned long long *list_count;
    uint32_t group_size;         // sequences per group (SHORT_G)
    uint32_t *gcounts;           // HIST_MODE 3: zeroed u32 rows of this wave (row 0 = sequence seq_base)
    unsigned long long *gtotals; // HIST_MODE 3: per-sequence window totals, zeroed (finalize_kernel reads them)
    uint64_t seq_base;           // HIST_MODE 3: first sequence of this wave
    uint64_t seq_count;          // HIST_MODE 3: sequences in this wave
    uint32_t tiles;              // HIST_MODE 3: CTAs cooperating on one sequence (work item = sequence x tile)
    const uint32_t *even_tab;    // HIST_MODE 7: [H*(H/32)] bitmap words then [H*(H/32)] u16 prefixes (see api.cu)
    uint32_t even_words;         // HIST_MODE 7: H*(H/32)
    uint32_t *out_list;          // HIST_MODE 5: sequences with > 65535 windows are appended here (next launch)
    unsigned long long *out_count;
};

// HIST_MODE 7 = rank space for EVEN k with the rank computed from two small shared-memory tables instead of a
//             4^k-entry table in L2 (mode 2 spends ~600 cycles of latency per k-mer on that look-up with only 8
//             warps per SM).  Write the code as (a, R), two halves of k/2 bases; it is canonical iff
//             a <= rc(R), so rank(a, R) = prefix[a][R/32] + popc(bitmap[a][R/32] & ((1 << R%32) - 1)) where
//             bitmap[a] marks the R' with rc(R') >= a.  k = 8: 8 KB + 4 KB of tables.
// HIST_MODE 5 = mode 7's in-kernel rank + 16-bit counters packed two to a word (rank r -> word r/2, half r&1):
//             k = 8 needs 64.25 KB + 12 KB instead of 128.5 KB + 12 KB, so two CTAs per SM can overlap their
//             accumulate and write-out phases.  Sequences with more than 65535 windows are passed on to a
//             second launch of mode 7 (out_list).
// HIST_MODE 4 = canonical, ODD k, dense half-size histogram: the two strands of an odd k-mer differ in the
//             top bit of their MIDDLE base (m vs 3-m), so "the strand whose middle base is A or C" is a
//             table-free representative; dropping that bit gives a dense index in [0, 4^k/2).  Half the
//             shared memory of mode 1 (k=7: 32 KB instead of 64 KB -> twice the CTAs per SM); the gather
//             table (canon_perm) maps rank -> this index.  Ranks whose representative is the reverse strand
//             would all fall into one bank (consecutive codes -> reverse complements that differ only in
//             their HIGH digits), so every row of 128 bins is skewed by one more word (k = 7 only).
// HIST_MODE 3 = histogram too large for shared memory: atomics (RED) go straight to the zeroed u32 row in
//             global memory / L2, index rank_full[f] (or f when rank_full is null); no write-out here.
// HIST_MODE: 0 = raw (index f), 1 = canonical code space (index min(f,r), gather on write-out),
//            2 = canonical rank space (index rank_full[f], linear write-out)
// count -> output element.  SMALL: every count (and the divisor) is below 2^23, so the float comes
// from the 2^23 magic constant (no quarter-rate I2F) and the exact f32 division sequence applies.
template <int OUT, bool NORM, bool SMALL>
__device__ __forceinline__ typename OutT<OUT>::type cvt_count(uint32_t cnt, float dF, float rinv, double dD) {
    if constexpr (OUT == OUT_U32) {
        return cnt;
    } else if constexpr (OUT == OUT_F32) {
        if constexpr (SMALL) {
            const float c = __uint_as_float(0x4B000000u | cnt) - 8388608.0f;
            return NORM ? quot_f32(c, dF, rinv) : c;
        } else {
            return NORM ? (float)((double)cnt / dD) : (float)cnt;
        }
    } else {
        return NORM ? (double)cnt / dD : (double)cnt;
    }
}

template <int OUT, int HIST_MODE, bool NORM, bool SMALL>
__device__ __forceinline__ void seq_write_row(uint32_t *hist, typename OutT<OUT>::type *row, const SeqParams &p,
                                              float dF, float rinv, double dD) {
    using T = typename OutT<OUT>::type;
    const uint32_t tid = threadIdx.x;
    // Code-space histograms are gathered through canon_of_rank.  Four consecutive ranks per lane would
    // stride the banks by ~8 words (codes are ~50 % dense): measured 4-way conflicts.  Instead lane l of
    // a warp takes ranks {l, 32+l, 64+l, 96+l} of a 128-rank block — consecutive across lanes, so the
    // monotone codes fall into distinct banks — fetched with ONE 128-bit load from a table permuted on
    // the host, and written back with four fully coalesced 32-bit stores.
    if constexpr (HIST_MODE == 5) {
        // rank space, 16-bit counters packed two to a word (rank r -> word r/2, half r&1): linear sweep, one
        // 128-bit shared load = 8 counts = two 128-bit (f32/u32) stores; zeroed on the way.  dim % 8 == 0.
        for (uint32_t w = tid * 4u; w < p.hist_entries; w += blockDim.x * 4u) {
            const uint4 hv = *reinterpret_cast<const uint4 *>(hist + w);
            *reinterpret_cast<uint4 *>(hist + w) = make_uint4(0, 0, 0, 0);
            const uint32_t hw[4] = {hv.x, hv.y, hv.z, hv.w};
            T e[8];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                e[2 * q] = cvt_count<OUT, NORM, SMALL>(hw[q] & 0xFFFFu, dF, rinv, dD);
                e[2 * q + 1] = cvt_count<OUT, NORM, SMALL>(hw[q] >> 16, dF, rinv, dD);
            }
            T *dst = row + 2u * w;
            if constexpr (OUT == OUT_F64) {
#pragma unroll
                for (int q = 0; q < 4; ++q) reinterpret_cast<double2 *>(dst)[q] = make_double2(e[2 * q], e[2 * q + 1]);
            } else if constexpr (OUT == OUT_F32) {
                reinterpret_cast<float4 *>(dst)[0] = make_float4(e[0], e[1], e[2], e[3]);
                reinterpret_cast<float4 *>(dst)[1] = make_float4(e[4], e[5], e[6], e[7]);
            } else {
                reinterpret_cast<uint4 *>(dst)[0] = make_uint4(e[0], e[1], e[2], e[3]);
                reinterpret_cast<uint4 *>(dst)[1] = make_uint4(e[4], e[5], e[6], e[7]);
            }
        }
        return;
    }
    if constexpr (HIST_MODE == 1 || HIST_MODE == 4) {
        const uint32_t nblk = p.dim >> 7;
        const uint32_t lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
        for (uint32_t b = warp; b < nblk; b += nwarps) {
            const uint4 cc = __ldg(reinterpret_cast<const uint4 *>(p.canon_perm + (b << 7)) + lane);
            const uint32_t c0 = hist[cc.x], c1 = hist[cc.y], c2 = hist[cc.z], c3 = hist[cc.w];
            hist[cc.x] = 0; hist[cc.y] = 0; hist[cc.z] = 0; hist[cc.w] = 0;
            T *dst = row + (b << 7) + lane;
            dst[0] = cvt_count<OUT, NORM, SMALL>(c0, dF, rinv, dD);
            dst[32] = cvt_count<OUT, NORM, SMALL>(c1, dF, rinv, dD);
            dst[64] = cvt_count<OUT, NORM, SMALL>(c2, dF, rinv, dD);
            dst[96] = cvt_count<OUT, NORM, SMALL>(c3, dF, rinv, dD);
        }
        for (uint32_t j = (nblk << 7) + tid; j < p.dim; j += blockDim.x) {  // ranks past the last full block
            const uint32_t cc = __ldg(p.canon_of_rank + j);
            const uint32_t cnt = hist[cc];
            hist[cc] = 0;
            row[j] = cvt_count<OUT, NORM, SMALL>(cnt, dF, rinv, dD);
        }
        return;
    }
    if (HIST_MODE != 1 && (p.dim & 3u) == 0) {
        for (uint32_t j = tid * 4u; j < p.dim; j += blockDim.x * 4u) {
            uint32_t cnt[4];
            if constexpr (HIST_MODE == 1) {
                const uint4 cc = __ldg(reinterpret_cast<const uint4 *>(p.canon_of_rank + j));
                cnt[0] = hist[cc.x]; cnt[1] = hist[cc.y]; cnt[2] = hist[cc.z]; cnt[3] = hist[cc.w];
                hist[cc.x] = 0; hist[cc.y] = 0; hist[cc.z] = 0; hist[cc.w] = 0;
            } else {
                const uint4 hv = *reinterpret_cast<const uint4 *>(hist + j);
                cnt[0] = hv.x; cnt[1] = hv.y; cnt[2] = hv.z; cnt[3] = hv.w;
                *reinterpret_cast<uint4 *>(hist + j) = make_uint4(0, 0, 0, 0);
            }
            const T e0 = cvt_count<OUT, NORM, SMALL>(cnt[0], dF, rinv, dD);
            const T e1 = cvt_count<OUT, NORM, SMALL>(cnt[1], dF, rinv, dD);
            const T e2 = cvt_count<OUT, NORM, SMALL>(cnt[2], dF, rinv, dD);
            const T e3 = cvt_count<OUT, NORM, SMALL>(cnt[3], dF, rinv, dD);
            if constexpr (OUT == OUT_F64) {
                reinterpret_cast<double2 *>(row + j)[0] = make_double2(e0, e1);
                reinterpret_cast<double2 *>(row + j)[1] = make_double2(e2, e3);
            } else if constexpr (OUT == OUT_F32) {
                *reinterpret_cast<float4 *>(row + j) = make_float4(e0, e1, e2, e3);
            } else {
                *reinterpret_cast<uint4 *>(row + j) = make_uint4(e0, e1, e2, e3);
            }
        }
    } else {
        for (uint32_t j = tid; j < p.dim; j += blockDim.x) {
            uint32_t cnt;
            if constexpr (HIST_MODE == 1) {
                const uint32_t cc = __ldg(p.canon_of_rank + j);
                cnt = hist[cc];
                hist[cc] = 0;
            } else {
                cnt = hist[j];
                hist[j] = 0;
            }
            row[j] = cvt_count<OUT, NORM, SMALL>(cnt, dF, rinv, dD);
        }
    }
}

// One CTA per sequence.  Warp w owns a contiguous range of the sequence's 16-base chunks and walks it
// 32 chunks per step; the look-back word of lane 0 is carried from lane 31 of the previous step (the
// first step is primed with the chunk before the range).  When every lane has 16 valid windows — the
// steady state — the 16 atomics are unconditional increments; otherwise each adds its validity bit.
// KT: compile-time k (0 = use p.k); the specialised instances fold the window-mask loop and every
// shift amount into immediates.
template <int OUT, int HIST_MODE, bool NORM, int KT = 0>
__global__ void __launch_bounds__((HIST_MODE == 2 || HIST_MODE == 7) ? 1024 : ((HIST_MODE == 5) ? 256 : KTB_SEQ_MAXTHREADS),
                                  (HIST_MODE == 2 || HIST_MODE == 7) ? 1 : (HIST_MODE == 5) ? 3 : ((HIST_MODE == 4) ? KTB_SEQ_MINBLOCKS4 : KTB_SEQ_MINBLOCKS))
seq_kernel(const SeqParams p) {
    extern __shared__ __align__(16) uint32_t hist[];
    __shared__ unsigned long long s_group;
    __shared__ uint32_t s_total[2];  // double-buffered so the reset never races a late reader

    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const uint32_t warp = tid >> 5;
    const uint32_t nwarps = blockDim.x >> 5;
    // work item = one sequence: (sequence of the wave, tile) in mode 3, else (group, index within the group) —
    // a whole group of 16 contigs per item left the last CTAs with megabases of work (19 % tail on config 4)
    const uint64_t nitems = (HIST_MODE == 3) ? p.seq_count * p.tiles
                            : (p.list ? (uint64_t)*p.list_count : (p.n + p.group_size - 1) / p.group_size) * p.group_size;
    if ((uint64_t)blockIdx.x >= nitems) return;  // nothing for this CTA (e.g. short_kernel took everything)
    for (uint32_t i = tid; i < p.hist_entries; i += blockDim.x) hist[i] = 0;
    // mode 7: rank tables behind the histogram (bitmap words, then u16 prefixes)
    uint32_t *s_bitmap = hist + ((p.hist_entries + 3u) & ~3u);
    uint16_t *s_prefix = reinterpret_cast<uint16_t *>(s_bitmap + p.even_words);
    if constexpr (HIST_MODE == 7 || HIST_MODE == 5) {
        for (uint32_t i = tid; i < p.even_words; i += blockDim.x) s_bitmap[i] = __ldg(p.even_tab + i);
        const uint16_t *gp = reinterpret_cast<const uint16_t *>(p.even_tab + p.even_words);
        if constexpr (HIST_MODE == 5) {   // every second prefix only: 2 KB less, which lets a third CTA fit on the SM
            for (uint32_t i = tid; i < p.even_words / 2; i += blockDim.x) s_prefix[i] = gp[2 * i];
        } else {
            for (uint32_t i = tid; i < p.even_words; i += blockDim.x) s_prefix[i] = gp[i];
        }
    }
    (void)s_bitmap; (void)s_prefix;
    if (tid == 0) { s_total[0] = 0; s_total[1] = 0; }
    __syncthreads();
    uint32_t it = 0;

    const uint32_t k = KT ? (uint32_t)KT : p.k;
    const uint32_t kmask4 = ((k >= 15) ? 0x3FFFFFFFu : ((1u << (2 * k)) - 1u)) << 2;  // code pre-scaled by 4
    const uint32_t midbit4 = 1u << (2 * (k / 2) + 1 + 2);  // top bit of the middle base (odd k), pre-scaled
    const uint32_t mb_shift = 2 * (k / 2) + 4;              // s4 >> mb_shift = digits above the middle bit
    const uint32_t mb_mul = midbit4 - 4u * (midbit4 >> 9);  // 2^m*4 minus the skew of 4 bytes per 128 bins
    (void)midbit4; (void)mb_shift; (void)mb_mul;
    using T = typename OutT<OUT>::type;
    T *out = reinterpret_cast<T *>(p.out);
    constexpr uint32_t FULL = 0xffffffffu;
    uint8_t *hbytes = reinterpret_cast<uint8_t *>(hist);
    const uint4 filler = make_uint4(0x41414141u, 0x41414141u, 0x41414141u, 0x41414141u);

    // p.grab consecutive items per trip to the work counter: one same-address atomic per 150-base read capped the
    // whole GPU at ~330 M reads/s; long sequences keep grab = 1 for the tail balance
    const unsigned long long grab = p.grab ? p.grab : 1u;
    for (;;) {
        if (tid == 0) s_group = atomicAdd(p.counter, grab);
        __syncthreads();
        const unsigned long long item0 = s_group;
        __syncthreads();  // everyone has read s_group before tid 0 overwrites it next round
        if (item0 >= nitems) break;
      for (unsigned long long item = item0; item < min(item0 + grab, (unsigned long long)nitems); ++item) {
        uint64_t i0;
        uint32_t nseq, tile = 0, tiles = 1;
        if constexpr (HIST_MODE == 3) {  // work item = (sequence of the wave, tile of that sequence)
            tiles = p.tiles;
            i0 = p.seq_base + item / tiles;
            tile = (uint32_t)(item % tiles);
            nseq = 1;
        } else {
            const uint64_t gi = item / p.group_size;
            const uint64_t g = p.list ? (uint64_t)p.list[gi] : gi;
            i0 = g * (uint64_t)p.group_size + (item - gi * p.group_size);
            nseq = (i0 < p.n) ? 1u : 0u;
        }

        for (uint32_t si = 0; si < nseq; ++si) {
            const uint64_t seq = i0 + si;
            const uint64_t s0 = p.offsets[seq];
            const uint64_t s1 = p.offsets[seq + 1];
            uint32_t mine = 0;  // valid windows counted by this thread
            if constexpr (HIST_MODE == 5) {
                if (s1 - s0 > 65535ull + k - 1) {   // a 16-bit counter could overflow: leave it to the next launch
                    if (tid == 0) p.out_list[atomicAdd(p.out_count, 1ULL)] = (uint32_t)seq;
                    continue;                        // uniform for the CTA; no barrier skipped inside this iteration
                }
            }
            if (s1 - s0 >= k) {
                const uint64_t cbase = s0 >> 4;                                     // absolute index of chunk 0
                const uint32_t nch = (uint32_t)(((s1 - 1) >> 4) - cbase) + 1u;      // chunks touching the sequence
                // whole 32-chunk steps are dealt out to the warps in contiguous runs (only the last step
                // of the sequence can be partial)
                const uint32_t nsteps = (nch + 31) >> 5;
                const uint32_t ts0 = (uint32_t)(((uint64_t)tile * nsteps) / tiles);        // this CTA's steps
                const uint32_t ts1 = (uint32_t)(((uint64_t)(tile + 1) * nsteps) / tiles);
                const uint32_t w0 = (ts0 + (warp * (ts1 - ts0)) / nwarps) << 5;
                const uint32_t w1 = min(nch, (ts0 + ((warp + 1) * (ts1 - ts0)) / nwarps) << 5);
                const uint32_t head_mask = 0xFFFFu >> (uint32_t)(s0 & 15);          // bases of chunk 0 inside the sequence
                const uint32_t tail_mask = ~(0xFFFFu >> ((uint32_t)((s1 - 1) & 15) + 1u)) & 0xFFFFu;
                if (w0 < w1) {
                    uint32_t carry_cf = 0, carry_vm = 0;
                    if (w0 > 0) {  // prime the look-back with the chunk before this warp's range
                        const uint4 v = load16_guarded(p.bases, (cbase + w0 - 1) << 4, p.total_bases);
                        decode16(v, carry_cf, carry_vm);
                        if (w0 == 1) carry_vm &= head_mask;
                    }
                    // only a sequence that ends within 16 bytes of the end of the buffer needs the guarded load
                    const uint4 *seq_chunks = reinterpret_cast<const uint4 *>(p.bases) + cbase;
                    const bool near_end = ((cbase + nch) << 4) > p.total_bases;
                    auto fetch = [&](uint32_t c) -> uint4 {
                        if (c >= w1) return filler;
                        if (near_end) return load16_guarded(p.bases, (cbase + c) << 4, p.total_bases);
                        return __ldg(seq_chunks + c);
                    };
                    uint4 vnext = fetch(w0 + lane);
                    for (uint32_t c0 = w0; c0 < w1; c0 += 32) {
                        const uint32_t c = c0 + lane;
                        const uint4 v = vnext;
                        if (c0 + 32 < w1) vnext = fetch(c + 32);  // prefetch the next step
                        uint32_t cf, vm;
                        decode16(v, cf, vm);
                        if (c >= w1) { vm = 0; cf = (uint32_t)lane * 0x9E3779B1u; }  // idle lanes add 0 at scattered bins
                        if (c == 0) vm &= head_mask;
                        if (c == nch - 1) vm &= tail_mask;
                        uint32_t cf_prev = __shfl_up_sync(FULL, cf, 1);
                        uint32_t vm_prev = __shfl_up_sync(FULL, vm, 1);
                        if (lane == 0) { cf_prev = carry_cf; vm_prev = carry_vm; }
                        carry_cf = __shfl_sync(FULL, cf, 31);
                        carry_vm = __shfl_sync(FULL, vm, 31);
                        // windows: bit b of vw set <=> V32 bits b..b+k-1 all set (older bases = higher bits)
                        const uint32_t vw = window_mask((vm_prev << 16) | vm, k) & 0xFFFFu;
                        mine += __popc(vw);
                        const uint64_t F64 = ((uint64_t)cf_prev << 32) | cf;
                        uint64_t R64 = 0;
                        if constexpr (HIST_MODE == 1 || HIST_MODE == 4 || HIST_MODE == 5 || HIST_MODE == 7) {
                            R64 = ((uint64_t)revcomp_pack(cf) << 32) | revcomp_pack(cf_prev);
                        }
                        uint32_t idx4[16];  // histogram byte offsets
#pragma unroll
                        for (int j = 0; j < 16; ++j) {
                            const uint32_t f4 = (j < 15) ? ((uint32_t)(F64 >> (2 * (14 - j))) & kmask4)
                                                         : ((cf << 2) & kmask4);
                            if constexpr (HIST_MODE == 0) {
                                idx4[j] = f4;
                            } else if constexpr (HIST_MODE == 1) {
                                const uint32_t r4 = (uint32_t)(R64 >> (2 * (16 + j - (int)k))) & kmask4;
                                idx4[j] = min(f4, r4);
                            } else if constexpr (HIST_MODE == 4) {
                                const uint32_t r4 = (uint32_t)(R64 >> (2 * (16 + j - (int)k))) & kmask4;
                                const uint32_t s4 = (f4 & midbit4) ? r4 : f4;          // strand with middle base A/C
                                // drop the (zero) middle bit AND skew rows of 128 bins by one word, in one IMAD:
                                // s = hi*2^(m+1) + lo  ->  d = hi*2^m + lo,  phys = d + (d >> 7 words) = s - hi*(2^m - 4)
                                const uint32_t hi = s4 >> mb_shift;
                                idx4[j] = s4 - hi * mb_mul;
                            } else if constexpr (HIST_MODE == 5) {
                                const uint32_t r4 = (uint32_t)(R64 >> (2 * (16 + j - (int)k))) & kmask4;
                                const uint32_t c = min(f4, r4) >> 2;
                                const uint32_t w = c >> 5;
                                const uint2 bw = reinterpret_cast<const uint2 *>(s_bitmap)[w >> 1];   // words w&~1, w|1
                                const bool odd = (w & 1u) != 0u;
                                const uint32_t below = (odd ? bw.y : bw.x) & ((1u << (c & 31u)) - 1u);
                                idx4[j] = (uint32_t)s_prefix[w >> 1] + (uint32_t)__popc(below) +
                                          (odd ? (uint32_t)__popc(bw.x) : 0u);   // rank; word/half split below
                            } else if constexpr (HIST_MODE == 7) {
                                const uint32_t r4 = (uint32_t)(R64 >> (2 * (16 + j - (int)k))) & kmask4;
                                const uint32_t c = min(f4, r4) >> 2;                 // canonical code (a, R)
                                const uint32_t w = c >> 5;                           // a * (H/32) + R / 32
                                const uint32_t below = s_bitmap[w] & ((1u << (c & 31u)) - 1u);
                                idx4[j] = ((uint32_t)s_prefix[w] + (uint32_t)__popc(below)) << 2;
                            } else if constexpr (HIST_MODE == 2) {
                                idx4[j] = __ldg(p.rank_full + (f4 >> 2)) << 2;
                            } else {
                                idx4[j] = p.rank_full ? (__ldg(p.rank_full + (f4 >> 2)) << 2) : f4;
                            }
                        }
                        if constexpr (HIST_MODE == 3) {
                            uint8_t *grow = reinterpret_cast<uint8_t *>(p.gcounts + (seq - p.seq_base) * (uint64_t)p.dim);
#pragma unroll
                            for (int j = 0; j < 16; ++j)
                                if (vw & (1u << (15 - j))) atomicAdd(reinterpret_cast<uint32_t *>(grow + idx4[j]), 1u);
                            continue;
                        }
                        if constexpr (HIST_MODE == 5) {
                            const bool all16 = __all_sync(FULL, vw == 0xFFFFu);
#pragma unroll
                            for (int j = 0; j < 16; ++j) {
                                const uint32_t rk = idx4[j];
                                const uint32_t one = all16 ? 1u : ((vw >> (15 - j)) & 1u);
                                atomicAdd(hist + (rk >> 1), one << ((rk & 1u) << 4));
                            }
                            continue;
                        }
                        if (KTB_SEQ_FASTPATH && __all_sync(FULL, vw == 0xFFFFu)) {
#pragma unroll
                            for (int j = 0; j < 16; ++j)
                                atomicAdd(reinterpret_cast<uint32_t *>(hbytes + idx4[j]), 1u);
                        } else {
#pragma unroll
                            for (int j = 0; j < 16; ++j)  // branch-free: an invalid window adds 0
                                atomicAdd(reinterpret_cast<uint32_t *>(hbytes + idx4[j]), (vw >> (15 - j)) & 1u);
                        }
                    }
                }
            }
            // ---- total = block sum of `mine`
#pragma unroll
            for (int s = 16; s > 0; s >>= 1) mine += __shfl_xor_sync(FULL, mine, s);
            if (lane == 0 && mine) atomicAdd(&s_total[it & 1], mine);
            __syncthreads();
            const uint32_t total = s_total[it & 1];
            if (tid == 0) s_total[(it + 1) & 1] = 0;  // slot of the next sequence; last read two barriers ago
            ++it;
            const uint64_t dv = norm_divisor(total, p.norm_mode, p.canonical);
            const float dF = (float)dv;
            const float rinv = __frcp_rn(dF);
            const double dD = (double)dv;
            if constexpr (HIST_MODE == 3) {
                if (tid == 0 && total) atomicAdd(p.gtotals + seq, (unsigned long long)total);
                __syncthreads();
                continue;
            }
            if (tid == 0 && p.totals) p.totals[seq] = total;
            // ---- write-out (normalisation fused), histogram re-zeroed on the way
            T *row = out + seq * (uint64_t)p.dim;
            if (dv < (1ULL << 23))
                seq_write_row<OUT, HIST_MODE, NORM, true>(hist, row, p, dF, rinv, dD);
            else
                seq_write_row<OUT, HIST_MODE, NORM, false>(hist, row, p, dF, rinv, dD);
            __syncthreads();
        }
      }
    }
}

// ================================================================================================
// wave_kernel — histograms larger than shared memory, ONE persistent cooperative launch
// ================================================================================================
// Same arithmetic as seq_kernel mode 3 (RED atomics straight into zeroed u32 rows), but the wave loop lives on
// the device.  A wave is a run of rows small enough that the wave being counted and the next one (zeroed at the
// end of the iteration) stay in L2 together, so a row reaches HBM once (ncu: DRAM writes = 1.1 x the output,
// reads = the bases).  Iteration w of every CTA:
//     step table of wave w  ->  RED the items of wave w  ->  [f32: grid barrier, normalise wave w in place]
//     ->  zero wave w+1  ->  grid barrier
// Work item = one 32-chunk step (512 bases) of one sequence, taken by a WARP; items are dealt round-robin over
// the CTAs so that every SM issues REDs: scattered REDs leave an SM at ~0.66 lanes/clock whatever the occupancy
// (tools/microbench_red.cu: 190 G/s chip-wide), which is the bound of the counting phase.
// Replaces ~3 launches per wave (row memset, counter memset, kernel) whose latency dominated the k = 10 path.
// Measured and NOT faster (profiles/r1k_wave_kernel_experiments.txt): flag-based split-phase barriers, warp-
// specialised zeroing with several waves in flight, prefetching the first item across the barrier, one zero
// store behind every RED.  A poll or dependent load queues behind the SM's own RED backlog, so every cross-SM
// hand-off costs microseconds, and zeroing ahead of the counting doubles the L2 footprint (about 64 MB is usable
// for this pattern), which halves the wave and doubles the number of barriers.
// Output u32 or f32 in place; f64 keeps the multi-launch path.
struct WaveParams {
    const uint8_t *bases;
    const uint64_t *offsets;
    uint64_t n;
    uint64_t total_bases;
    uint32_t *rows;               // n x dim u32 (u32 / f32 output written in place)
    unsigned long long *totals;   // n, zeroed before the launch
    const uint32_t *rank_full;    // RANK 1: [4^k]
    const uint32_t *rank_tab;     // RANK 2: canonical-code bitmap (tab_words) + u32 prefix per PAIR of words
    uint32_t tab_words;
    uint64_t dim;
    uint64_t wave_rows;           // sequences per wave (<= 256)
    uint32_t k;
    int norm_mode;
    int canonical;
};

// zero rows [s0, s1): thread `t` of `nt`
__device__ __forceinline__ void wave_zero_rows(const WaveParams &p, uint64_t s0, uint64_t s1, uint64_t t, uint64_t nt) {
    if (s0 >= s1) return;
    uint4 *dst = reinterpret_cast<uint4 *>(p.rows + s0 * p.dim);
    const uint64_t nvec = (s1 - s0) * p.dim / 4;   // dim % 4 == 0 on this path
    for (uint64_t i = t; i < nvec; i += nt) dst[i] = make_uint4(0, 0, 0, 0);
}

__device__ __forceinline__ float4 wave_cvt4(const WaveParams &p, uint4 c, unsigned long long total) {
    const bool norm = p.norm_mode != NORM_COUNTS;
    const uint64_t dv = norm_divisor(total, p.norm_mode, p.canonical);
    const float dF = (float)dv, rinv = __frcp_rn(dF);
    const double dD = (double)dv;
    float4 o;
    if (!norm) {   // a count is at most `total`: the magic-constant conversion is exact below 2^23
        if (total < (1ULL << 23)) {
            o.x = cvt_count<OUT_F32, false, true>(c.x, dF, rinv, dD);
            o.y = cvt_count<OUT_F32, false, true>(c.y, dF, rinv, dD);
            o.z = cvt_count<OUT_F32, false, true>(c.z, dF, rinv, dD);
            o.w = cvt_count<OUT_F32, false, true>(c.w, dF, rinv, dD);
        } else {
            o.x = cvt_count<OUT_F32, false, false>(c.x, dF, rinv, dD);
            o.y = cvt_count<OUT_F32, false, false>(c.y, dF, rinv, dD);
            o.z = cvt_count<OUT_F32, false, false>(c.z, dF, rinv, dD);
            o.w = cvt_count<OUT_F32, false, false>(c.w, dF, rinv, dD);
        }
    } else if (dv < (1ULL << 23)) {
        o.x = cvt_count<OUT_F32, true, true>(c.x, dF, rinv, dD);
        o.y = cvt_count<OUT_F32, true, true>(c.y, dF, rinv, dD);
        o.z = cvt_count<OUT_F32, true, true>(c.z, dF, rinv, dD);
        o.w = cvt_count<OUT_F32, true, true>(c.w, dF, rinv, dD);
    } else {
        o.x = cvt_count<OUT_F32, true, false>(c.x, dF, rinv, dD);
        o.y = cvt_count<OUT_F32, true, false>(c.y, dF, rinv, dD);
        o.z = cvt_count<OUT_F32, true, false>(c.z, dF, rinv, dD);
        o.w = cvt_count<OUT_F32, true, false>(c.w, dF, rinv, dD);
    }
    return o;
}

// counts -> f32 in place for rows [s0, s1): thread `t` of `nt`, 2 independent 16-byte loads in flight per thread.
// The row of a vector (for its total) is tracked incrementally: one 64-bit division per thread, not per vector.
__device__ __forceinline__ void wave_finalize_rows(const WaveParams &p, uint64_t s0, uint64_t s1, uint64_t t, uint64_t nt) {
    if (s0 >= s1) return;
    constexpr int U = 2;
    const uint64_t vpr = p.dim / 4;                 // vectors per row (dim % 4 == 0 on this path)
    const uint64_t nvec = (s1 - s0) * vpr;
    const uint64_t dq = nt / vpr, dr = nt % vpr;    // one stride of nt vectors = dq rows + dr vectors
    uint64_t row = t / vpr, col = t % vpr;          // of vector i0
    uint4 *buf = reinterpret_cast<uint4 *>(p.rows + s0 * p.dim);
    for (uint64_t i0 = t; i0 < nvec; i0 += U * nt) {
        uint4 c[U];
        unsigned long long tot[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const uint64_t i = i0 + (uint64_t)u * nt;
            if (i < nvec) {
                c[u] = __ldcg(buf + i);
                tot[u] = __ldcg(p.totals + s0 + row);
            }
            row += dq;
            col += dr;
            if (col >= vpr) { col -= vpr; ++row; }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const uint64_t i = i0 + (uint64_t)u * nt;
            if (i < nvec) reinterpret_cast<float4 *>(buf)[i] = wave_cvt4(p, c[u], tot[u]);
        }
    }
}

// RANK: 0 raw codes, 1 rank through the L2-resident table, 2 rank computed from shared-memory tables (one
// look-up + RED per k-mer through L2 halves to the RED alone; the tables fit up to k = 10).
template <int RANK, bool F32>
__global__ void __launch_bounds__(1024) wave_kernel(const WaveParams p) {
    namespace cg = cooperative_groups;
    cg::grid_group grid = cg::this_grid();
    extern __shared__ __align__(16) uint32_t s_tab[];   // RANK 2: bitmap words, then pair prefixes
    __shared__ uint32_t s_steps[256 + 1];   // exclusive prefix of 32-chunk steps per sequence of the wave (<= 256 rows)
    __shared__ uint32_t s_wsum[8];
    if constexpr (RANK == 2) {
        const uint32_t nw = p.tab_words + p.tab_words / 2;
        for (uint32_t i = threadIdx.x; i < nw; i += blockDim.x) s_tab[i] = __ldg(p.rank_tab + i);
    }
    const uint32_t *s_prefix = s_tab + p.tab_words;
    (void)s_prefix;
    __syncthreads();

    const int tid = threadIdx.x, lane = tid & 31;
    const uint32_t k = p.k;
    const uint32_t kmask = (1u << (2 * k)) - 1u;
    constexpr uint32_t FULL = 0xffffffffu;
    const uint32_t G = gridDim.x;
    const uint64_t slot = (uint64_t)(tid >> 5) * G + blockIdx.x;   // consecutive items on different SMs
    const uint64_t nslots = (uint64_t)G * (blockDim.x >> 5);
    const uint64_t gt = (uint64_t)blockIdx.x * blockDim.x + tid, gnt = (uint64_t)G * blockDim.x;
    const uint64_t nwaves = (p.n + p.wave_rows - 1) / p.wave_rows;
    const uint4 filler = make_uint4(0x41414141u, 0x41414141u, 0x41414141u, 0x41414141u);
    auto wave_lo = [&](uint64_t w) { return min(p.n, w * p.wave_rows); };

    // step table of wave w into s_steps; returns the number of (sequence, step) items.  All threads call.
    auto build_table = [&](uint64_t w) -> uint32_t {
        const uint64_t s0 = wave_lo(w);
        const uint32_t rows = (uint32_t)(wave_lo(w + 1) - s0);
        uint32_t *tab = s_steps;
        uint32_t mysteps = 0;
        if ((uint32_t)tid < rows) {
            const uint64_t a = p.offsets[s0 + tid], b = p.offsets[s0 + tid + 1];
            const uint32_t nch = (b - a >= k) ? (uint32_t)(((b - 1) >> 4) - (a >> 4)) + 1u : 0u;
            mysteps = (nch + 31) >> 5;
        }
        uint32_t incl = mysteps;   // inclusive scan over the first 256 threads
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t t = __shfl_up_sync(FULL, incl, d);
            if (lane >= d) incl += t;
        }
        if (lane == 31 && tid < 256) s_wsum[tid >> 5] = incl;
        __syncthreads();
        if (tid < 256) {
            uint32_t base = 0;
            for (int ww = 0; ww < (tid >> 5); ++ww) base += s_wsum[ww];
            tab[tid + 1] = base + incl;
        }
        if (tid == 0) tab[0] = 0;
        __syncthreads();
        return tab[rows];
    };
    // one item: find its (sequence, step) in the table, load 16 bases per lane, RED the windows that end in them
    auto do_item = [&](uint64_t w, uint32_t item) {
        const uint64_t s0 = wave_lo(w);
        const uint32_t rows = (uint32_t)(wave_lo(w + 1) - s0);
        uint32_t lo = 0, hi = rows;   // largest r with s_steps[r] <= item
        while (hi - lo > 1) {
            const uint32_t mid = (lo + hi) >> 1;
            if (s_steps[mid] <= item) lo = mid; else hi = mid;
        }
        const uint64_t seq = s0 + lo;
        const uint32_t step = item - s_steps[lo];
        const uint64_t q0 = p.offsets[seq], q1 = p.offsets[seq + 1];
        const uint64_t cbase = q0 >> 4;
        const uint32_t nch = (uint32_t)(((q1 - 1) >> 4) - cbase) + 1u;
        const uint32_t c = step * 32u + lane;
        const uint4 v = (c < nch) ? load16_guarded(p.bases, (cbase + c) << 4, p.total_bases) : filler;
        // the chunk before this step belongs to another warp's item: re-read it for the windows that straddle
        const uint4 vp = (lane == 0 && c > 0) ? load16_guarded(p.bases, (cbase + c - 1) << 4, p.total_bases) : filler;
        uint32_t cf, vm;
        decode16(v, cf, vm);
        if (c >= nch) vm = 0;
        if (c == 0) vm &= 0xFFFFu >> (uint32_t)(q0 & 15);
        if (c == nch - 1) vm &= ~(0xFFFFu >> ((uint32_t)((q1 - 1) & 15) + 1u)) & 0xFFFFu;
        uint32_t cf_prev = __shfl_up_sync(FULL, cf, 1);
        uint32_t vm_prev = __shfl_up_sync(FULL, vm, 1);
        if (lane == 0) {
            cf_prev = 0; vm_prev = 0;
            if (c > 0) {
                decode16(vp, cf_prev, vm_prev);
                if (c - 1 == 0) vm_prev &= 0xFFFFu >> (uint32_t)(q0 & 15);
            }
        }
        const uint32_t vw = window_mask((vm_prev << 16) | vm, k) & 0xFFFFu;
        uint32_t cnt = __popc(vw);
        const uint64_t F64 = ((uint64_t)cf_prev << 32) | cf;
        uint32_t *row = p.rows + seq * p.dim;
        uint32_t idx[16];   // all 16 ranks before the first RED (f is always a valid code, also for invalid windows)
        uint64_t R64 = 0;
        if constexpr (RANK == 2) R64 = ((uint64_t)revcomp_pack(cf) << 32) | revcomp_pack(cf_prev);
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            const uint32_t f = (uint32_t)(F64 >> (2 * (15 - j))) & kmask;
            if constexpr (RANK == 0) {
                idx[j] = f;
            } else if constexpr (RANK == 1) {
                idx[j] = __ldg(p.rank_full + f);
            } else {
                const uint32_t r = (uint32_t)(R64 >> (2 * (17 + j - (int)k))) & kmask;
                const uint32_t cc = min(f, r);
                const uint32_t wd = cc >> 5;
                const uint2 bw = reinterpret_cast<const uint2 *>(s_tab)[wd >> 1];
                const bool odd = (wd & 1u) != 0u;
                const uint32_t below = (odd ? bw.y : bw.x) & ((1u << (cc & 31u)) - 1u);
                idx[j] = s_prefix[wd >> 1] + (uint32_t)__popc(below) + (odd ? (uint32_t)__popc(bw.x) : 0u);
            }
        }
#pragma unroll
        for (int j = 0; j < 16; ++j)
            if (vw & (1u << (15 - j))) atomicAdd(row + idx[j], 1u);
#pragma unroll
        for (int sft = 16; sft > 0; sft >>= 1) cnt += __shfl_xor_sync(FULL, cnt, sft);
        if (lane == 0 && cnt) atomicAdd(p.totals + seq, (unsigned long long)cnt);
    };

    wave_zero_rows(p, 0, wave_lo(1), gt, gnt);
    grid.sync();
    for (uint64_t w = 0; w < nwaves; ++w) {
        const uint32_t nitems = build_table(w);
        for (uint64_t item = slot; item < nitems; item += nslots) {
            do_item(w, (uint32_t)item);
        }
        // f32: normalise the wave in place as soon as all its REDs have landed (a second barrier per wave is cheaper
        // than keeping a third wave in L2 until the next iteration: 6.4 ms -> see DESIGN.md §4.3)
        if constexpr (F32) {
            grid.sync();
            wave_finalize_rows(p, wave_lo(w), wave_lo(w + 1), gt, gnt);
        }
        // u32: warps without an item start here at once, so the zeroing overlaps the REDs of the others; the zeroed
        // wave only has to stay in L2 from now on, which is why a wave can be as large as a third of L2
        wave_zero_rows(p, wave_lo(w + 1), wave_lo(w + 2), gt, gnt);
        grid.sync();
    }
}

// ================================================================================================
// flat_kernel — flat decomposition of the base stream + global atomics (any k <= 12)
// ================================================================================================
struct FlatParams {
    const uint8_t *bases;
    const uint64_t *offsets;
    uint64_t n;
    uint64_t total_bases;
    uint32_t *counts;            // n x dim, zeroed
    unsigned long long *totals;  // n, zeroed
    const uint32_t *rank_full;   // [4^k] or nullptr in raw mode
    uint64_t dim;
    uint32_t k;
};

constexpr int FLAT_CHUNK = 32;

__global__ void __launch_bounds__(256) flat_kernel(const FlatParams p) {
    const uint32_t k = p.k;
    const uint32_t kmask = (k >= 16) ? 0xFFFFFFFFu : ((1u << (2 * k)) - 1u);
    const uint64_t nchunks = (p.total_bases + FLAT_CHUNK - 1) / FLAT_CHUNK;
    for (uint64_t ch = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; ch < nchunks;
         ch += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t p0 = ch * FLAT_CHUNK;
        const uint64_t p1 = min(p0 + (uint64_t)FLAT_CHUNK, p.total_bases);
        // sequence containing p0: largest s with offsets[s] <= p0 < offsets[s+1]
        uint64_t lo = 0, hi = p.n;  // invariant: offsets[lo] <= p0, offsets[hi] > p0 (offsets[n] = total > p0)
        while (hi - lo > 1) {
            const uint64_t mid = (lo + hi) >> 1;
            if (p.offsets[mid] <= p0) lo = mid; else hi = mid;
        }
        uint64_t s = lo;
        uint64_t s_end = p.offsets[s + 1];
        const uint64_t s_begin = p.offsets[s];
        uint64_t q = (p0 >= (uint64_t)(k - 1)) ? p0 - (k - 1) : 0;
        if (q < s_begin) q = s_begin;
        uint32_t f = 0, run = 0;
        unsigned long long tot = 0;
        for (uint64_t pos = q; pos < p1; ++pos) {
            while (pos >= s_end) {  // crossed into the next (possibly empty) sequence
                if (tot) { atomicAdd(p.totals + s, tot); tot = 0; }
                ++s;
                s_end = p.offsets[s + 1];
                run = 0;
            }
            const uint32_t c = nt4_code(p.bases[pos]);
            f = ((f << 2) | (c & 3u)) & kmask;
            run = (c < 4u) ? run + 1u : 0u;
            if (run >= k && pos >= p0) {
                const uint32_t idx = p.rank_full ? __ldg(p.rank_full + f) : f;
                atomicAdd(p.counts + s * p.dim + idx, 1u);
                ++tot;
            }
        }
        if (tot) atomicAdd(p.totals + s, tot);
    }
}

// counts (u32, n x dim) -> out (n x dim of OUT); in place when OUT is 4 bytes wide and out == counts
template <int OUT>
__global__ void __launch_bounds__(256) finalize_kernel(const uint32_t *counts, const unsigned long long *totals,
                                                       void *outv, uint64_t *totals_out, uint64_t n,
                                                       uint64_t dim, int norm_mode, int canonical) {
    using T = typename OutT<OUT>::type;
    T *out = reinterpret_cast<T *>(outv);
    const bool norm = norm_mode != NORM_COUNTS;
    const uint64_t nel = n * dim;
    for (uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; e < nel;
         e += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t s = e / dim;
        const unsigned long long total = totals[s];
        const uint64_t dv = norm_divisor(total, norm_mode, canonical);
        const bool small_div = dv < (1ULL << 24);
        const float dF = (float)dv;
        out[e] = make_out<OUT>(counts[e], norm, small_div, dF, __frcp_rn(dF), (double)dv);
        if (totals_out && e == s * dim) totals_out[s] = total;
    }
}

}  // namespace ktb
