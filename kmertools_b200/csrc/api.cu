// api.cu — host side of the C ABI declared in include/kmertools_b200.h.
//
// Mirrors the reference's OligoComputer life cycle (composition/src/oligo.rs:31-93,
// pybindings/src/oligo.rs:22-99): create = build the kmer_pos_maps tables once, vectorise = run the
// per-sequence histogram + normalisation for a whole batch.  No CPU compute path exists here: without
// a CUDA device every compute entry point returns KTB_ERR_NODEVICE.
#include "../../include/kmertools_b200.h"
#include "device_guard.h"
#include "kernels.cuh"
#include "long_kernel.cuh"
#include "bucket_kernels.cuh"

#include <algorithm>
#include <chrono>
#include <climits>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

// The module declares the kernels' extern __shared__ arrays in the order the kernels are first instantiated, and a
// kernel's dynamic shared memory starts at the strictest alignment declared up to its own array.  Instantiating these
// two first keeps the histograms of seq_kernel and short_kernel 16 bytes after their static variables (not 128, as
// behind long_kernel's and count_kernel's arrays) whatever order the launchers below are written in.
template __global__ void ktb::seq_kernel<ktb::OUT_U32, 3, false>(ktb::SeqParams);
template __global__ void ktb::short_kernel<ktb::OUT_U32, false>(ktb::ShortParams);

void ktb_internal_register_host(void *p, size_t bytes);   // multi.cu: registry of page-locked blocks
void ktb_internal_free_host(void *p);

namespace {

thread_local std::string g_err;

int fail(int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}

#define CU(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess)                                                                     \
            return fail(e_ == cudaErrorMemoryAllocation ? KTB_ERR_NOMEM : KTB_ERR_CUDA,            \
                        "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

uint64_t rev_comp(uint64_t x, int k) {  // kmer/src/kmer.rs:43-52
    uint64_t r = 0;
    for (int i = 0; i < k; ++i) {
        r = (r << 2) | ((x & 3) ^ 3);
        x >>= 2;
    }
    return r;
}

struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    DevBuf() = default;
    DevBuf(const DevBuf &) = delete;
    DevBuf &operator=(const DevBuf &) = delete;
    ~DevBuf() {
        if (p) cudaFree(p);
    }
    int ensure(size_t bytes) {
        if (bytes <= cap) return KTB_OK;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        size_t want = bytes + bytes / 8 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) {
            e = cudaMalloc(&p, bytes);
            want = bytes;
        }
        if (e != cudaSuccess) {
            p = nullptr;
            return fail(KTB_ERR_NOMEM, "cudaMalloc(%zu) failed: %s", bytes, cudaGetErrorString(e));
        }
        cap = want;
        return KTB_OK;
    }
};

constexpr int NBUF = 3;

struct ChunkSet {
    cudaStream_t stream = nullptr;
    cudaEvent_t ev[5] = {};  // h2d start/end, kernel end, d2h end, kernel start
    DevBuf bases, offsets, out, totals;
    bool busy = false;
};

}  // namespace

struct ktb_oligo {
    int k = 0;
    int device = 0;
    uint64_t ncodes = 0;  // 4^k
    uint64_t dim_canon = 0;
    std::vector<uint32_t> rank_of_canon;   // [4^k] canonical code -> rank, 0 elsewhere (pos_map)
    std::vector<uint32_t> canon_of_rank;   // [dim_canon]
    // device tables
    uint32_t *d_rank_full = nullptr;       // [4^k] any code -> rank of its canonical form
    uint32_t *d_canon_of_rank = nullptr;   // [dim_canon padded to 4]
    uint32_t *d_canon_perm = nullptr;      // canon_of_rank permuted inside 128-rank blocks (seq_kernel gather)
    uint32_t *d_mb_of_rank = nullptr;      // odd k: rank -> dense middle-base index (seq_kernel mode 4)
    uint32_t *d_mb_perm = nullptr;
    uint32_t *d_even_tab = nullptr;        // even k: bitmap words + u16 prefixes for the in-kernel rank (mode 7)
    uint32_t even_words = 0;
    uint32_t *d_wave_tab = nullptr;        // canonical-code bitmap + u32 pair prefixes for wave_kernel<2>
    uint32_t wave_tab_words = 0;
    bool wave_tab_in_smem = false;         // the whole table fits shared memory (wave_kernel RANK 2)
    bool wave_seg_aligned = false;         // every 2^13-code segment starts at a column that is a multiple of 4
    uint64_t mb_entries = 0;               // histogram words mode 4 needs (dense index + skew)
    uint32_t *d_k7_sched = nullptr;        // k = 7: conflict-free write-out schedule of long_kernel MODE_K7
    uint32_t *d_fwd_sched = nullptr;       // 3 <= k <= 6: (offset of c | offset of rc(c) << 16) per rank, long_kernel MODE_FWD
    uint32_t *d_short_tab_canon = nullptr; // [4^k] (k <= 5): (word byte offset << 22) | 8*(bin&3)
    uint32_t *d_short_tab_raw = nullptr;
    unsigned long long *d_counters = nullptr;  // [4]
    DevBuf ws_totals, ws_counts, ws_list, ws_list2, ws_order;
    DevBuf ws_tiles, ws_pool, ws_runs, ws_wavectr;   // bucket path: tile prefix + records, sorted code pool, run descriptors, work counters
    std::vector<cudaEvent_t> wave_ev;      // bucket path: bucket_kernel(w) done
    ChunkSet sets[NBUF];
    cudaStream_t aux[2] = {nullptr, nullptr};   // wave overlap in the global-atomic path
    cudaEvent_t aux_ev[3] = {nullptr, nullptr, nullptr};
    cudaEvent_t ref_ev = nullptr;            // time origin of the stats of one host-buffer call
    int sm_count = 0;
    size_t smem_optin = 0;
    // options
    int64_t chunk_bytes = 512ll << 20;
    int force_path = 0;
    int seq_threads = 0;  // 0 = auto (256)
    int seq_grab = 0;     // work items per atomic in seq_kernel (0 = from the mean sequence length)
    int dense_odd = 1;    // use seq_kernel mode 4 where it applies
    int even_rank = 1;    // use seq_kernel mode 7 where it applies
    int long_warps = 0;   // warps per CTA of long_kernel: 0 = from the mean sequence length, else 4 or 8
    int k7_mid = 1;       // long_kernel MODE_K7 (k = 7 canonical, u32 / f32 rows)
    int fwd_replicas = 1; // MODE_FWD on long contigs: lane-private replicas of the bins (k <= 5)
    int fwd_fold = 1;     // long_kernel MODE_FWD (3 <= k <= 6 canonical, long sequences, u32 / f32 rows)
    int64_t fwd_min_len = 1024;   // mean sequence length from which MODE_FWD replaces seq_kernel mode 1
    int bucket = 1;       // rows larger than shared memory: bucket_kernel + count_kernel instead of global atomics
    int k8_long = 1;            // k = 8 (packed 16-bit rank-space histogram): long_kernel MODE_K8 instead of seq_kernel mode 5
    int longest_first = 1;      // long contigs (replica variants of long_kernel): hand out the long sequences first
    int bucket_hist_kb = 64;    // histogram memory of count_kernel per CTA: 64 KB (three CTAs per SM) or 96 KB (two)
    int bucket_wave_ctas = 2;   // bucket_kernel CTAs per SM when the path runs in waves (beside count_kernel's three)
    int bucket_waves = 1;       // waves of that path (bucket_kernel of wave w+1 overlaps count_kernel of wave w); measured: 1 is best
    int bucket_log2_seg = 14;   // columns per segment of that path (2^14 u32 bins = 64 KB of shared memory)
    int packed16 = 1;     // seq_kernel mode 5 (k = 8: packed 16-bit rank-space histogram, 2 CTAs/SM)
    int global_steps_per_warp = 1;
    int wave_persistent = 1;                 // global-atomic path as one cooperative launch (u32 / f32 output)
    bool coop_launch = false;                // device attribute, read at create
    int64_t wave_budget_bytes = 96ll << 20;  // L2 budget of the cooperative kernel, a wave is a third of it
    int wave_smem_rank = 1;                  // rank from shared-memory tables when they fit (k <= 10)
    int64_t global_wave_bytes = 64ll << 20;  // rows zeroed + counted together in the global-atomic path (fits L2)
    ktb_stats stats{};
};

namespace {

using namespace ktb;

using ktb::DeviceGuard;
#define ON_DEVICE(dev)                                                                              \
    DeviceGuard device_guard_(dev);                                                                 \
    if (device_guard_.err != cudaSuccess)                                                           \
        return fail(KTB_ERR_CUDA, "cudaSetDevice(%d) failed: %s", (int)(dev), cudaGetErrorString(device_guard_.err))

template <typename K>
int set_smem(K kern, size_t bytes) {
    CU(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    return KTB_OK;
}

// Grid of a launch: the CTAs of `kern` that fit the GPU at once (at most `max_per_sm` per SM), no more than `items`,
// and at least one.
template <typename K>
int fit_grid(const ktb_oligo *h, K kern, int threads, size_t smem, uint64_t items, unsigned *grid,
             int max_per_sm = INT_MAX) {
    int per_sm = 1;
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, threads, smem));
    per_sm = std::max(1, std::min(per_sm, max_per_sm));
    *grid = (unsigned)std::max<uint64_t>(1, std::min<uint64_t>((uint64_t)h->sm_count * per_sm, items));
    return KTB_OK;
}

// Checks the launches just enqueued and counts them in the stats of the call.
int launched(ktb_oligo *h, int count = 1) {
    CU(cudaGetLastError());
    h->stats.launches += count;
    return KTB_OK;
}

// Work items per trip to the (same-address) work counter: one atomic per 150-base read capped the GPU at ~330 M
// reads/s, so short sequences take several; long sequences keep one item per trip for the tail.
uint32_t grab(const ktb_oligo *h, uint64_t mean_len) {
    return h->seq_grab > 0 ? (uint32_t)h->seq_grab
                           : (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(16, 4096 / std::max<uint64_t>(mean_len, 1)));
}

// The batch of one call: device inputs and outputs, the row width and the caller's stream.
struct Batch {
    const uint8_t *bases;
    const uint64_t *offsets;
    uint64_t n, total_bases, dim;
    int canonical, norm_mode;
    void *out;
    uint64_t *totals;
    cudaStream_t st;
};

struct ShortCfg {
    bool ok = false;
    uint32_t words = 0, max_len = 0;
    size_t smem = 0;
};

constexpr int SHORT_WARPS = 8;

ShortCfg short_config(const ktb_oligo *h, uint64_t dim) {
    ShortCfg c;
    if (h->ncodes > (uint64_t)SHORT_MAX_CODES || (dim & 3) || h->force_path != 0) return c;
    c.words = (uint32_t)(dim / 4);
    c.max_len = 254u + (uint32_t)h->k;
    c.smem = (size_t)SHORT_WARPS * ((size_t)SHORT_G * c.words + SHORT_PAD) * 4;
    c.ok = c.smem + 8192 <= h->smem_optin;
    return c;
}

template <int OUT>
int launch_short(ktb_oligo *h, const Batch &b, const ShortCfg &c) {
    ShortParams p{};
    p.ngroups = (b.n + SHORT_G - 1) / SHORT_G;
    if (int rc = h->ws_list.ensure(p.ngroups * 4)) return rc;
    p.bases = b.bases; p.offsets = b.offsets; p.n = b.n;
    p.total_bases = b.total_bases;
    p.out = b.out; p.totals = b.totals;
    p.tab = b.canonical ? h->d_short_tab_canon : h->d_short_tab_raw;
    p.counter = h->d_counters + 0;
    p.reject_list = (uint32_t *)h->ws_list.p;
    p.reject_count = h->d_counters + 2;
    p.k = h->k; p.ncodes = (uint32_t)h->ncodes; p.dim = (uint32_t)b.dim; p.words = c.words;
    p.words_recip = c.words > 1 ? (uint32_t)(0xFFFFFFFFu / c.words + 1u) : 0u;
    p.max_len = c.max_len;
    p.norm_mode = b.norm_mode; p.canonical = b.canonical;
    auto kern = (p.norm_mode != NORM_COUNTS) ? short_kernel<OUT, true> : short_kernel<OUT, false>;
    if (int rc = set_smem(kern, c.smem)) return rc;
    unsigned grid;
    if (int rc = fit_grid(h, kern, SHORT_WARPS * 32, c.smem, (p.ngroups + SHORT_WARPS - 1) / SHORT_WARPS, &grid)) return rc;
    kern<<<grid, SHORT_WARPS * 32, c.smem, b.st>>>(p);
    return launched(h);
}

template <int OUT>
int launch_seq(ktb_oligo *h, SeqParams p, int hist_mode, cudaStream_t st) {
    const size_t smem = (hist_mode == 5) ? ((((size_t)p.hist_entries + 3) & ~(size_t)3) * 4 + (size_t)p.even_words * 5 + 16)
                        : (hist_mode == 7) ? ((((size_t)p.hist_entries + 3) & ~(size_t)3) * 4 + (size_t)p.even_words * 6 + 16)
                                         : (size_t)p.hist_entries * 4;
    void (*kern)(const SeqParams) = nullptr;
    const bool nrm = p.norm_mode != NORM_COUNTS;
    if (hist_mode == 0) kern = nrm ? seq_kernel<OUT, 0, true> : seq_kernel<OUT, 0, false>;
    else if (hist_mode == 1) kern = nrm ? seq_kernel<OUT, 1, true> : seq_kernel<OUT, 1, false>;
    else if (hist_mode == 4) kern = nrm ? seq_kernel<OUT, 4, true> : seq_kernel<OUT, 4, false>;
    else if (hist_mode == 5) kern = nrm ? seq_kernel<OUT, 5, true> : seq_kernel<OUT, 5, false>;
    else if (hist_mode == 7) kern = nrm ? seq_kernel<OUT, 7, true> : seq_kernel<OUT, 7, false>;
    else kern = nrm ? seq_kernel<OUT, 2, true> : seq_kernel<OUT, 2, false>;
    if constexpr (OUT == OUT_F32) {
        if (hist_mode == 4 && nrm && p.k == 7) kern = seq_kernel<OUT_F32, 4, true, 7>;   // k folded into immediates for the headline shapes
        if (hist_mode == 1 && nrm) {
            switch (p.k) {
                case 4: kern = seq_kernel<OUT_F32, 1, true, 4>; break;
                case 5: kern = seq_kernel<OUT_F32, 1, true, 5>; break;
                case 6: kern = seq_kernel<OUT_F32, 1, true, 6>; break;
                case 7: kern = seq_kernel<OUT_F32, 1, true, 7>; break;
                default: break;
            }
        }
    }
    if (int rc = set_smem(kern, smem)) return rc;
    // measured (bench.py --seq-threads): 10 kbp reads with a <= 16 KB histogram run 20 % faster with 4 warps
    // per CTA (less barrier / priming overhead, occupancy is not the limit); long contigs and the big
    // histograms want 8 warps.
    const uint64_t mean_len = p.total_bases / std::max<uint64_t>(p.n, 1);
    const int auto_threads = (mean_len <= 512 && smem <= 16 * 1024 && hist_mode != 5) ? 64   // one step per read: k = 6 short reads +7 %
                             : ((mean_len <= 16384 && (smem <= 16 * 1024 || hist_mode == 5)) ? 128 : 256);
    int threads = h->seq_threads > 0 ? h->seq_threads : auto_threads;
    if (hist_mode == 5 && threads > 256) threads = 256;
    if (hist_mode != 2 && hist_mode != 5 && hist_mode != 7 && threads > KTB_SEQ_MAXTHREADS) threads = KTB_SEQ_MAXTHREADS;
    const uint64_t nitems = ((p.n + p.group_size - 1) / p.group_size) * p.group_size;   // one sequence per item
    unsigned grid;
    if (int rc = fit_grid(h, kern, threads, smem, nitems, &grid)) return rc;
    p.grab = grab(h, mean_len);
    kern<<<grid, threads, smem, st>>>(p);
    return launched(h);
}

// Splits the (bin word, rank) pairs of a row into groups of 32 whose source banks (word % 32) are all distinct and
// whose destination banks (rank % 32) are all distinct, so that a warp moves a group between two shared-memory
// arrays without a bank conflict on either side.  The pairs are the edges of a bipartite multigraph (source bank,
// destination bank) that is d-regular with d = n / 32; when d is a power of two it is split into two d/2-regular
// halves by alternating along closed trails (every vertex keeps half of its edges on each side) until d = 1, i.e.
// perfect matchings.  `word_of_rank[j]` must be a bijection onto [0, n); returns the ranks group after group, lane
// l of a group holding the pair whose rank has bank l.  Empty on failure (n / 32 not a power of two).
std::vector<uint32_t> conflict_free_groups(const std::vector<uint32_t> &word_of_rank) {
    const uint32_t n = (uint32_t)word_of_rank.size();
    if (n == 0 || n % 32) return {};
    const uint32_t deg = n / 32;
    if (deg & (deg - 1)) return {};
    std::vector<std::vector<uint32_t>> parts(1), next;
    parts[0].resize(n);
    for (uint32_t j = 0; j < n; ++j) parts[0][j] = j;
    for (uint32_t d = deg; d > 1; d >>= 1) {
        next.clear();
        for (const auto &edges : parts) {
            // adjacency: vertices 0..31 = source banks, 32..63 = destination banks
            std::vector<uint32_t> adj[64];
            for (uint32_t e = 0; e < edges.size(); ++e) {
                adj[word_of_rank[edges[e]] & 31].push_back(e);
                adj[32 + (edges[e] & 31)].push_back(e);
            }
            std::vector<uint8_t> used(edges.size(), 0);
            size_t ptr[64] = {};
            std::vector<uint32_t> half[2];
            for (int v0 = 0; v0 < 64; ++v0) {
                int cur = v0, side = 0;
                for (;;) {
                    while (ptr[cur] < adj[cur].size() && used[adj[cur][ptr[cur]]]) ++ptr[cur];
                    if (ptr[cur] == adj[cur].size()) break;   // only possible back at v0: every degree is even
                    const uint32_t e = adj[cur][ptr[cur]];
                    used[e] = 1;
                    half[side].push_back(edges[e]);
                    side ^= 1;
                    const int a = (int)(word_of_rank[edges[e]] & 31), b = 32 + (int)(edges[e] & 31);
                    cur = (cur == a) ? b : a;
                }
            }
            if (half[0].size() != half[1].size()) return {};
            next.push_back(std::move(half[0]));
            next.push_back(std::move(half[1]));
        }
        parts.swap(next);
    }
    std::vector<uint32_t> order(n);
    for (size_t g = 0; g < parts.size(); ++g) {
        if (parts[g].size() != 32) return {};
        uint32_t seen_s = 0, seen_d = 0;
        for (uint32_t j : parts[g]) {
            seen_s |= 1u << (word_of_rank[j] & 31);
            seen_d |= 1u << (j & 31);
            order[g * 32 + (j & 31)] = j;
        }
        if (seen_s != 0xFFFFFFFFu || seen_d != 0xFFFFFFFFu) return {};
    }
    return order;
}

// long_kernel over the groups on `list` (every group when it is null) in `mode`.
template <int OUT>
int launch_long(ktb_oligo *h, const Batch &b, int mode, const uint32_t *list, unsigned long long *list_count) {
    if constexpr (OUT == OUT_F64) {
        (void)h; (void)b; (void)mode; (void)list; (void)list_count;
        return fail(KTB_ERR_ARG, "long_kernel has no f64 instance");
    } else {
        LongParams p{};
        p.bases = b.bases; p.offsets = b.offsets; p.n = b.n; p.total_bases = b.total_bases;
        p.out = b.out; p.totals = b.totals;
        p.counter = h->d_counters + 1;
        p.list = list; p.list_count = list_count;
        p.group_shift = 4;   // SHORT_G
        static_assert(SHORT_G == 16, "group_shift");
        p.k = h->k; p.dim = (uint32_t)b.dim;
        p.norm_mode = b.norm_mode; p.canonical = b.canonical;
        if (mode == MODE_K8) {
            // the packed 16-bit rank-space histogram of seq_kernel mode 5; sequences it cannot count go on out_list
            p.even_tab = h->d_even_tab; p.even_words = h->even_words;
            p.out_list = (uint32_t *)h->ws_list2.p; p.out_count = h->d_counters + 3;
            p.hist_words = (uint32_t)(h->dim_canon / 2);
        } else {
            p.sched = mode == MODE_K7 ? h->d_k7_sched : h->d_fwd_sched;
            p.hist_words = mode == MODE_K7 ? K7_BINS : (uint32_t)h->ncodes + 4;
        }
        const bool nrm = p.norm_mode != NORM_COUNTS;
        const uint64_t mean_len = p.total_bases / std::max<uint64_t>(p.n, 1);
        // 4 warps per CTA for reads of a few steps per warp (10 kbp = 20 steps: 5 per warp, balanced, half the per-warp
        // set-up of 8 warps); 8 warps for long contigs
        // measured (profiles/r2_sweeps.txt): k = 7 rows ran best with 10 warps per CTA (three CTAs per SM of 64 KB each)
        // until the kernel looked ahead across sequences; that needs 72 registers, which 8 warps have and 10 do not
        // (799 against 765 Gbases/s on config 3, 20.6 against 18.6 on 150-base reads).  The small histograms of k <= 5 run
        // best with 4 warps
        int nw = h->long_warps > 0 ? h->long_warps : (mode == MODE_K7 ? 8 : (mode == MODE_K8 ? (mean_len <= 16384 ? 4 : 8) : (mean_len <= 32768 ? 4 : 8)));
        if (nw == 10 && mode != MODE_K7) nw = 8;
        void (*kern)(const LongParams) = nullptr;
        int rs = 0;
        if (mode == MODE_K8) {
            if (nw != 8) nw = 4;
            if (nw == 4) kern = nrm ? long_kernel<OUT, true, MODE_K8, 4> : long_kernel<OUT, false, MODE_K8, 4>;
            else kern = nrm ? long_kernel<OUT, true, MODE_K8, 8> : long_kernel<OUT, false, MODE_K8, 8>;
        } else if (mode == MODE_K7) {
            if (nw == 4) kern = nrm ? long_kernel<OUT, true, MODE_K7, 4> : long_kernel<OUT, false, MODE_K7, 4>;
            else if (nw == 10) kern = nrm ? long_kernel<OUT, true, MODE_K7, 10> : long_kernel<OUT, false, MODE_K7, 10>;
            else kern = nrm ? long_kernel<OUT, true, MODE_K7, 8> : long_kernel<OUT, false, MODE_K7, 8>;
        } else {
            if (nw == 4) kern = nrm ? long_kernel<OUT, true, MODE_FWD, 4> : long_kernel<OUT, false, MODE_FWD, 4>;
            else kern = nrm ? long_kernel<OUT, true, MODE_FWD, 8> : long_kernel<OUT, false, MODE_FWD, 8>;
            // long contigs at k <= 5: lane-private replicas of the (few) bins, k folded into immediates
            if (h->fwd_replicas && mean_len >= 32768 && nw == 8) {
                if (p.k == 3) { kern = nrm ? long_kernel<OUT, true, MODE_FWD, 8, 3, 5> : long_kernel<OUT, false, MODE_FWD, 8, 3, 5>; rs = 5; }
                if (p.k == 4) { kern = nrm ? long_kernel<OUT, true, MODE_FWD, 8, 4, 5> : long_kernel<OUT, false, MODE_FWD, 8, 4, 5>; rs = 5; }
                if (p.k == 5) { kern = nrm ? long_kernel<OUT, true, MODE_FWD, 8, 5, 3> : long_kernel<OUT, false, MODE_FWD, 8, 5, 3>; rs = 3; }
            }
        }
        if (rs) p.hist_words = (((uint32_t)1 << (2 * p.k)) << rs) + (1u << rs);   // + the always-zero replicas (rc slot of palindromes)
        const size_t smem = mode == MODE_K8 ? ((((size_t)p.hist_words + 3) & ~(size_t)3) * 4 + (size_t)p.even_words * 5 + 16)
                                            : ((((size_t)p.hist_words + 31) & ~(size_t)31) + p.dim) * 4;
        if (int rc = set_smem(kern, smem)) return rc;
        const int threads = nw * 32;
        const uint64_t nitems = ((p.n + SHORT_G - 1) / SHORT_G) * SHORT_G;
        unsigned grid;
        if (int rc = fit_grid(h, kern, threads, smem, nitems, &grid)) return rc;
        p.grab = grab(h, mean_len);
        if (rs && h->longest_first && p.n > grid && p.n < (1ull << 32)) {
            // more contigs than CTAs: the queue order decides how long the last CTA runs alone (see order_count_kernel)
            if (int rc = h->ws_order.ensure(p.n * 4 + 129 * 8 + 64)) return rc;
            OrderParams op{};
            op.offsets = p.offsets; op.n = p.n; op.list = p.list; op.list_count = p.list_count; op.group_shift = p.group_shift;
            op.cls = (unsigned long long *)h->ws_order.p;
            op.order = (uint32_t *)((uint8_t *)h->ws_order.p + 129 * 8 + 56);
            CU(cudaMemsetAsync(op.cls, 0, 129 * 8, b.st));
            const unsigned ogrid = (unsigned)std::min<uint64_t>((nitems + 255) / 256, (uint64_t)h->sm_count * 4);
            order_count_kernel<<<ogrid, 256, 0, b.st>>>(op);
            order_scatter_kernel<<<ogrid, 256, 0, b.st>>>(op);
            if (int rc = launched(h, 2)) return rc;
            p.list = op.order; p.list_count = op.cls + 128; p.group_shift = 0;
            p.grab = 1;
        }
        kern<<<grid, threads, smem, b.st>>>(p);
        return launched(h);
    }
}

// u32 counts of rows [i0, i0 + cnt) -> normalised output rows (the counts are the u32 output itself)
template <int OUT>
int launch_finalize(ktb_oligo *h, const Batch &b, const uint32_t *counts, const unsigned long long *tot, uint64_t i0,
                    uint64_t cnt, cudaStream_t st) {
    if (OUT == OUT_U32) return KTB_OK;
    const size_t esize = (OUT == OUT_F64) ? 8 : 4;
    const unsigned grid = (unsigned)std::min<uint64_t>((cnt * b.dim + 255) / 256, (uint64_t)h->sm_count * 16);
    finalize_kernel<OUT><<<grid, 256, 0, st>>>(counts, tot + i0, (uint8_t *)b.out + i0 * b.dim * esize, nullptr, cnt,
                                               b.dim, b.norm_mode, b.canonical);
    return launched(h);
}

// Bucket-then-count (bucket_kernels.cuh): partition the k-mer codes of every tile by their high bits, then count each
// (sequence, code segment) in shared memory and write its part of the row once.  Writes the totals itself.
template <int OUT>
int launch_bucket(ktb_oligo *h, const Batch &b, unsigned long long *tot, uint64_t nseg) {
    const uint32_t log2_seg = (uint32_t)h->bucket_log2_seg;
    const uint64_t n = b.n, total_bases = b.total_bases;
    const cudaStream_t st = b.st;
    const uint64_t tile_bases = (uint64_t)BK_TILE_CHUNKS * 16;
    const uint64_t ntiles_bound = total_bases / tile_bases + 2 * n + 2;
    if (ntiles_bound >= (1ull << 31)) return fail(KTB_ERR_ARG, "batch too large for the bucket path");
    if (int rc = h->ws_tiles.ensure((n + 1) * 4 + 64 + ntiles_bound * sizeof(TileInfo))) return rc;
    if (int rc = h->ws_pool.ensure(ntiles_bound * (uint64_t)BK_TILE_CAP * 2 + 64)) return rc;
    if (int rc = h->ws_runs.ensure(ntiles_bound * nseg * 4)) return rc;
    uint32_t *tile_prefix = (uint32_t *)h->ws_tiles.p;
    TileInfo *tiles = (TileInfo *)((uint8_t *)h->ws_tiles.p + (((n + 1) * 4 + 63) & ~(uint64_t)63));
    tile_prefix_kernel<<<1, 1024, 0, st>>>(b.offsets, n, (uint32_t)h->k, tile_prefix);
    tile_info_kernel<<<(unsigned)std::min<uint64_t>((ntiles_bound + 255) / 256, (uint64_t)h->sm_count * 8), 256, 0, st>>>(
        b.offsets, n, tile_prefix, tiles);
    if (int rc = launched(h, 2)) return rc;
    BucketParams bp{};
    bp.bases = b.bases; bp.n = n; bp.total_bases = total_bases;
    bp.tile_prefix = tile_prefix; bp.tiles = tiles;
    bp.pool = (uint16_t *)h->ws_pool.p; bp.runs = (uint32_t *)h->ws_runs.p; bp.totals = tot;
    bp.k = (uint32_t)h->k; bp.nseg = (uint32_t)nseg; bp.log2_seg = log2_seg;
    CountParams cp{};
    cp.tile_prefix = tile_prefix; cp.pool = bp.pool; cp.runs = bp.runs; cp.totals_in = tot;
    cp.totals_out = b.totals; cp.out = b.out;
    cp.rank_tab = h->d_wave_tab; cp.tab_words = h->wave_tab_words;
    cp.n = n; cp.dim = b.dim; cp.nseg = (uint32_t)nseg; cp.log2_seg = log2_seg;
    cp.norm_mode = b.norm_mode; cp.canonical = b.canonical;
#ifdef KTB_COUNT_PROBE
    if (const char *e = getenv("KTB_COUNT_PROBE")) cp.probe = (uint32_t)atoi(e);
#endif
    void (*bkern)(const BucketParams) = b.canonical ? bucket_kernel<true> : bucket_kernel<false>;
    if (b.canonical && log2_seg == 14) {   // the two shapes BASELINE.json names get their constants at compile time
        if (h->k == 10) bkern = bucket_kernel<true, 10, 14>;
        else if (h->k == 9) bkern = bucket_kernel<true, 9, 14>;
    }
    const bool nrm = b.norm_mode != NORM_COUNTS;
    void (*ckern)(const CountParams) =
        b.canonical ? (nrm ? count_kernel<OUT, true, true> : count_kernel<OUT, false, true>)
                    : (nrm ? count_kernel<OUT, true, false> : count_kernel<OUT, false, false>);
    // histogram memory: 64 KB either way — one buffer of 2^14 bins (segments with at most half as many columns
    // alternate between its halves) or two buffers of 2^13
    const size_t S = (size_t)1 << log2_seg;
    cp.hist_words = (uint32_t)(log2_seg < 14 ? 2 * S : S);
    if (h->bucket_hist_kb == 96) cp.hist_words = 24576;   // segments of up to 12,288 columns alternate between two halves
    const size_t csmem = ((size_t)cp.hist_words + 2 * (S / 32)) * 4;
    if (int rc = set_smem(ckern, csmem)) return rc;
    // Waves (option "bucket_waves", default 1): bucket_kernel is bound by the integer pipe, count_kernel by latency and
    // the row writes, so the batch can be cut into waves with bucket_kernel(w+1) on one helper stream and
    // count_kernel(w) on the other, sharing the SMs.  Measured on config 5ii (profiles/r2_sweeps.txt, batch r2i):
    // 1.57 ms with one wave, 1.63 - 1.77 ms with 2 - 16 — the two kernels take each other's shared memory and
    // registers and both lose more occupancy than the overlap returns.  Kept as an option.
    const uint64_t nchunks = (n + CK_SEQ_CHUNK - 1) / CK_SEQ_CHUNK;
    const uint64_t nwaves = std::max<uint64_t>(1, std::min<uint64_t>((uint64_t)std::max(1, h->bucket_waves), nchunks / 16));
    if (int rc = h->ws_wavectr.ensure(nwaves * sizeof(unsigned long long))) return rc;
    CU(cudaMemsetAsync(h->ws_wavectr.p, 0, nwaves * sizeof(unsigned long long), st));
    CU(cudaEventRecord(h->aux_ev[2], st));
    cudaStream_t sb = nwaves > 1 ? h->aux[0] : st, sc = nwaves > 1 ? h->aux[1] : st;
    if (nwaves > 1) {
        CU(cudaStreamWaitEvent(sb, h->aux_ev[2], 0));
        CU(cudaStreamWaitEvent(sc, h->aux_ev[2], 0));
    }
    const int b_ctas = nwaves > 1 ? h->bucket_wave_ctas : INT_MAX;   // beside count_kernel when the waves overlap
    for (uint64_t w = 0; w < nwaves; ++w) {
        const uint64_t c_lo = nchunks * w / nwaves, c_hi = nchunks * (w + 1) / nwaves;
        bp.seq_lo = std::min(n, c_lo * CK_SEQ_CHUNK); bp.seq_hi = std::min(n, c_hi * CK_SEQ_CHUNK);
        const uint64_t wave_tiles = (bp.seq_hi - bp.seq_lo) * 2 + (total_bases / tile_bases) / nwaves + 2;   // grid bound only
        unsigned grid;
        if (int rc = fit_grid(h, bkern, BK_WARPS * 32, 0, wave_tiles, &grid, b_ctas)) return rc;
        bkern<<<grid, BK_WARPS * 32, 0, sb>>>(bp);
        if (int rc = launched(h)) return rc;
        if (nwaves > 1) {
            if (h->wave_ev.size() <= w) {
                cudaEvent_t e = nullptr;
                CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
                h->wave_ev.push_back(e);
            }
            CU(cudaEventRecord(h->wave_ev[w], sb));
            CU(cudaStreamWaitEvent(sc, h->wave_ev[w], 0));
        }
        cp.chunk_lo = c_lo; cp.chunk_hi = c_hi;
        cp.counter = (unsigned long long *)h->ws_wavectr.p + w;
        if (int rc = fit_grid(h, ckern, CK_THREADS, csmem, (c_hi - c_lo) * nseg, &grid)) return rc;
        ckern<<<grid, CK_THREADS, csmem, sc>>>(cp);
        if (int rc = launched(h)) return rc;
    }
    if (nwaves > 1) {
        CU(cudaEventRecord(h->aux_ev[0], sb));
        CU(cudaEventRecord(h->aux_ev[1], sc));
        CU(cudaStreamWaitEvent(st, h->aux_ev[0], 0));
        CU(cudaStreamWaitEvent(st, h->aux_ev[1], 0));
    }
    return KTB_OK;
}

// The flat-decomposition fallback (testing, force_path 1): the whole batch at once.
template <int OUT>
int launch_flat(ktb_oligo *h, const Batch &b, unsigned long long *tot) {
    const uint64_t row_bytes = b.dim * 4;
    uint32_t *counts = (uint32_t *)b.out;
    if (OUT == OUT_F64) {
        if (int rc = h->ws_counts.ensure(b.n * row_bytes)) return rc;
        counts = (uint32_t *)h->ws_counts.p;
    }
    CU(cudaMemsetAsync(counts, 0, b.n * row_bytes, b.st));
    if (b.total_bases > 0) {
        FlatParams fp{};
        fp.bases = b.bases; fp.offsets = b.offsets; fp.n = b.n; fp.total_bases = b.total_bases;
        fp.counts = counts; fp.totals = tot;
        fp.rank_full = b.canonical ? h->d_rank_full : nullptr;
        fp.dim = b.dim; fp.k = h->k;
        const uint64_t nchunks = (b.total_bases + FLAT_CHUNK - 1) / FLAT_CHUNK;
        const unsigned grid = (unsigned)std::min<uint64_t>((nchunks + 255) / 256, (uint64_t)h->sm_count * 32);
        flat_kernel<<<grid, 256, 0, b.st>>>(fp);
        if (int rc = launched(h)) return rc;
    }
    return launch_finalize<OUT>(h, b, counts, tot, 0, b.n, b.st);
}

// One persistent cooperative launch: the wave loop (zero next rows / count / normalise previous rows) runs on the
// device with a grid barrier per wave instead of three launches per wave.
template <int OUT>
int launch_wave_kernel(ktb_oligo *h, const Batch &b, unsigned long long *tot) {
    WaveParams wp{};
    wp.bases = b.bases; wp.offsets = b.offsets; wp.n = b.n; wp.total_bases = b.total_bases;
    wp.rows = (uint32_t *)b.out; wp.totals = tot;
    wp.rank_full = b.canonical ? h->d_rank_full : nullptr;
    wp.dim = b.dim; wp.k = (uint32_t)h->k; wp.norm_mode = b.norm_mode; wp.canonical = b.canonical;
    // a wave is a third of the budget: the wave being counted and the next one (zeroed at the end of the
    // iteration) are live together, the rest is slack for lines on their way out (32 MB waves measured best)
    wp.wave_rows = std::max<uint64_t>(1, std::min<uint64_t>(256, (uint64_t)h->wave_budget_bytes / 3 / (b.dim * 4)));
    const int rank_mode = !b.canonical ? 0 : (h->d_wave_tab && h->wave_tab_in_smem && h->wave_smem_rank) ? 2 : 1;
    wp.rank_tab = h->d_wave_tab; wp.tab_words = h->wave_tab_words;
    constexpr bool F32 = (OUT == OUT_F32);
    const void *kern = rank_mode == 0 ? (const void *)wave_kernel<0, F32>
                     : rank_mode == 1 ? (const void *)wave_kernel<1, F32> : (const void *)wave_kernel<2, F32>;
    const int threads = 1024;
    const size_t smem = rank_mode == 2 ? ((size_t)h->wave_tab_words * 6 + 16) : 0;
    if (smem > 48 * 1024) CU(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 1;
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, threads, smem));
    if (per_sm < 1) return fail(KTB_ERR_CUDA, "wave_kernel does not fit on an SM (%zu bytes of shared memory)", smem);
    const unsigned grid = (unsigned)h->sm_count;   // one CTA per SM: the RED rate of an SM does not grow with occupancy
    void *args[] = {&wp};
    CU(cudaLaunchCooperativeKernel(kern, dim3(grid), dim3(threads), args, smem, b.st));
    h->stats.launches++;
    return KTB_OK;
}

// Waves of rows that fit L2 together: zero the wave's rows, let every CTA of the GPU work on that wave (sequences
// are split into tiles), normalise it, move on.  The REDs then hit rows that are still L2-resident and each row goes
// to HBM once; one big memset + one launch over the whole batch made every RED a 32-byte DRAM read-modify-write
// (measured 8.5 ms vs the 0.7 ms roofline).
template <int OUT>
int launch_wave_loop(ktb_oligo *h, const Batch &b, unsigned long long *tot) {
    const uint64_t n = b.n, dim = b.dim, row_bytes = dim * 4;
    SeqParams qp{};
    qp.bases = b.bases; qp.offsets = b.offsets; qp.n = n; qp.total_bases = b.total_bases;
    qp.rank_full = b.canonical ? h->d_rank_full : nullptr;
    qp.counter = h->d_counters + 1;
    qp.k = h->k; qp.dim = (uint32_t)dim; qp.hist_entries = 0;
    qp.norm_mode = b.norm_mode; qp.canonical = b.canonical;
    qp.list = nullptr; qp.list_count = nullptr; qp.group_size = 1;
    qp.gtotals = tot;
    auto kern = seq_kernel<OUT_U32, 3, false>;
    // mode 3 is compiled for at most KTB_SEQ_MAXTHREADS threads: a larger CTA would not launch
    const int threads = std::min(h->seq_threads > 0 ? h->seq_threads : 128, KTB_SEQ_MAXTHREADS);
    // two waves in flight (one per helper stream), each half of the L2 budget
    const uint64_t wave = std::max<uint64_t>(1, std::min<uint64_t>(n, (uint64_t)h->global_wave_bytes / 2 / row_bytes));
    if (OUT == OUT_F64)
        if (int rc = h->ws_counts.ensure(2 * wave * row_bytes)) return rc;
    // a work item = (sequence, tile).  A wave is small (rows must fit L2), so parallelism has to come from
    // splitting sequences finely: about `global_steps_per_warp` steps of 512 bases per warp (the first
    // version used 4 and ran 5 warps per SM; one step per warp fills the machine).
    const uint64_t mean_steps = (b.total_bases / std::max<uint64_t>(n, 1)) / 512 + 1;
    const uint64_t per_item = (uint64_t)std::max(1, h->global_steps_per_warp) * (threads / 32);
    const uint32_t tiles = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(4096, mean_steps / per_item));
    CU(cudaEventRecord(h->aux_ev[2], b.st));
    uint64_t w = 0;
    for (uint64_t i0 = 0; i0 < n; i0 += wave, ++w) {
        const int x = (int)(w & 1);
        cudaStream_t sx = h->aux[x];
        if (w < 2) CU(cudaStreamWaitEvent(sx, h->aux_ev[2], 0));
        const uint64_t cnt = std::min(wave, n - i0);
        uint32_t *counts = (OUT == OUT_F64) ? (uint32_t *)h->ws_counts.p + (uint64_t)x * wave * dim
                                            : (uint32_t *)b.out + i0 * dim;
        CU(cudaMemsetAsync(counts, 0, cnt * row_bytes, sx));
        CU(cudaMemsetAsync(h->d_counters + 4 + x, 0, sizeof(unsigned long long), sx));
        qp.counter = h->d_counters + 4 + x;
        qp.gcounts = counts; qp.seq_base = i0; qp.seq_count = cnt; qp.tiles = tiles;
        unsigned grid;
        if (int rc = fit_grid(h, kern, threads, 0, cnt * tiles, &grid)) return rc;
        kern<<<grid, threads, 0, sx>>>(qp);
        if (int rc = launched(h)) return rc;
        if (int rc = launch_finalize<OUT>(h, b, counts, tot, i0, cnt, sx)) return rc;
    }
    for (int x = 0; x < 2; ++x) {   // join the helper streams back into the caller's stream
        CU(cudaEventRecord(h->aux_ev[x], h->aux[x]));
        CU(cudaStreamWaitEvent(b.st, h->aux_ev[x], 0));
    }
    return KTB_OK;
}

// Which histogram of seq_kernel fits shared memory (its mode), and its entries; -1 when none does.
int smem_hist_mode(const ktb_oligo *h, int canonical, uint64_t *entries) {
    const size_t smem_limit = h->smem_optin - 1024;
    if (h->force_path == 1) return -1;
    if (!canonical) {
        if (h->ncodes * 4 <= smem_limit) { *entries = h->ncodes; return 0; }
    } else if ((h->k & 1) && h->ncodes * 4 > 32 * 1024 && h->ncodes * 2 <= 64 * 1024 && h->dense_odd) {
        *entries = (h->mb_entries + 3) & ~3ull; return 4;   // k = 7: dense middle-base index, 32 KB + skew
    } else if (h->ncodes * 4 <= 64 * 1024) {
        *entries = h->ncodes; return 1;
    } else if (h->d_even_tab && h->even_rank && h->packed16 && (h->dim_canon % 8) == 0 &&
               h->dim_canon * 2 + h->even_words * 6 + 64 <= smem_limit / 2) {
        *entries = h->dim_canon / 2; return 5;   // k = 8: packed 16-bit rank space, 2 CTAs/SM
    } else if (h->d_even_tab && h->even_rank && h->dim_canon * 4 + h->even_words * 6 + 64 <= smem_limit) {
        *entries = h->dim_canon; return 7;      // k = 8: rank from shared-memory bitmap tables
    } else if (h->dim_canon * 4 <= smem_limit) {
        *entries = h->dim_canon; return 2;
    }
    return -1;
}

template <int OUT>
int run_device(ktb_oligo *h, const Batch &b) {
    if (b.n == 0) return KTB_OK;
    uint64_t hist_entries = 0;
    const int hist_mode = smem_hist_mode(h, b.canonical, &hist_entries);
    if (hist_mode >= 0) {
        CU(cudaMemsetAsync(h->d_counters, 0, 4 * sizeof(unsigned long long), b.st));
        const ShortCfg sc = short_config(h, b.dim);
        if (sc.ok)
            if (int rc = launch_short<OUT>(h, b, sc)) return rc;
        // the CTA-per-sequence kernels take the groups the short kernel rejected, or every group when it did not run
        const uint32_t *list = sc.ok ? (const uint32_t *)h->ws_list.p : nullptr;
        unsigned long long *list_count = sc.ok ? h->d_counters + 2 : nullptr;
        // second-generation CTA-per-sequence kernel (long_kernel.cuh) where it applies
        const bool long_ok = OUT != OUT_F64 && b.canonical && h->force_path != 3;
        const uint64_t mean_len = b.total_bases / std::max<uint64_t>(b.n, 1);
        if (long_ok && h->k == 7 && h->k7_mid && h->d_k7_sched) return launch_long<OUT>(h, b, MODE_K7, list, list_count);
        if (long_ok && h->d_fwd_sched && h->fwd_fold && (int64_t)mean_len >= h->fwd_min_len)
            return launch_long<OUT>(h, b, MODE_FWD, list, list_count);
        SeqParams qp{};
        qp.bases = b.bases; qp.offsets = b.offsets; qp.n = b.n; qp.total_bases = b.total_bases;
        qp.out = b.out; qp.totals = b.totals;
        qp.rank_full = h->d_rank_full;
        qp.canon_of_rank = hist_mode == 4 ? h->d_mb_of_rank : h->d_canon_of_rank;
        qp.canon_perm = hist_mode == 4 ? h->d_mb_perm : h->d_canon_perm;
        qp.counter = h->d_counters + 1;
        qp.k = h->k; qp.dim = (uint32_t)b.dim; qp.hist_entries = (uint32_t)hist_entries;
        qp.norm_mode = b.norm_mode; qp.canonical = b.canonical;
        qp.list = list; qp.list_count = list_count;
        qp.group_size = SHORT_G;
        qp.even_tab = h->d_even_tab; qp.even_words = h->even_words;
        if (hist_mode != 5) return launch_seq<OUT>(h, qp, hist_mode, b.st);
        // packed 16-bit counters: sequences with more than 65535 windows come back on out_list and are
        // redone with 32-bit counters (mode 7) in a second launch
        if (int rc = h->ws_list2.ensure(b.n * 4)) return rc;
        qp.out_list = (uint32_t *)h->ws_list2.p; qp.out_count = h->d_counters + 3;
        if (long_ok && h->k8_long && h->k == 8) {
            // same arithmetic inside long_kernel's loop (look-back lane, look-ahead across sequences)
            if (int rc = launch_long<OUT>(h, b, MODE_K8, list, list_count)) return rc;
        } else if (int rc = launch_seq<OUT>(h, qp, 5, b.st)) return rc;
        qp.hist_entries = (uint32_t)h->dim_canon;
        qp.counter = h->d_counters + 0;   // unused by the short kernel for this k, zeroed above
        qp.list = (const uint32_t *)h->ws_list2.p; qp.list_count = h->d_counters + 3; qp.group_size = 1;
        return launch_seq<OUT>(h, qp, 7, b.st);
    }

    // ---- rows larger than shared memory: zeroed u32 rows in HBM/L2, RED atomics, finalize
    if (int rc = h->ws_totals.ensure(b.n * 8)) return rc;
    unsigned long long *tot = (unsigned long long *)h->ws_totals.p;
    CU(cudaMemsetAsync(tot, 0, b.n * 8, b.st));
    const uint64_t nseg = (h->ncodes + (1ull << h->bucket_log2_seg) - 1) >> h->bucket_log2_seg;
    if (h->bucket && h->force_path == 0 && nseg <= (uint64_t)BK_MAX_SEG && (b.dim & 3) == 0 && h->k <= 10 &&
        (!b.canonical || (h->d_wave_tab && h->wave_seg_aligned)) && b.n < (1ull << 31) && b.total_bases < (1ull << 44))
        return launch_bucket<OUT>(h, b, tot, nseg);
    const int rc = h->force_path == 1 ? launch_flat<OUT>(h, b, tot)
                 : (h->wave_persistent && h->coop_launch && OUT != OUT_F64) ? launch_wave_kernel<OUT>(h, b, tot)
                 : launch_wave_loop<OUT>(h, b, tot);
    if (rc) return rc;
    if (b.totals) CU(cudaMemcpyAsync(b.totals, tot, b.n * 8, cudaMemcpyDeviceToDevice, b.st));
    return KTB_OK;
}

int dispatch_device(ktb_oligo *h, const uint8_t *d_bases, const uint64_t *d_offsets, uint64_t n,
                    uint64_t total_bases, int canonical, int norm_mode, int out_dtype, void *d_out,
                    uint64_t *d_totals, cudaStream_t st) {
    const Batch b{d_bases, d_offsets, n, total_bases, canonical ? h->dim_canon : h->ncodes, canonical, norm_mode,
                  d_out, d_totals, st};
    switch (out_dtype) {
        case KTB_OUT_U32: return run_device<OUT_U32>(h, b);
        case KTB_OUT_F32: return run_device<OUT_F32>(h, b);
        default: return run_device<OUT_F64>(h, b);
    }
}

}  // namespace

// internal (hidden) entry points shared with file_api.cu
__attribute__((visibility("hidden"))) int ktb_internal_dispatch(ktb_oligo *h, const uint8_t *d_bases,
                                                               const uint64_t *d_offsets, uint64_t n,
                                                               uint64_t total_bases, int canonical, int norm_mode,
                                                               int out_dtype, void *d_out, uint64_t *d_totals,
                                                               cudaStream_t st) {
    ON_DEVICE(h->device);
    return dispatch_device(h, d_bases, d_offsets, n, total_bases, canonical, norm_mode, out_dtype, d_out, d_totals, st);
}
__attribute__((visibility("hidden"))) int ktb_internal_fail(int code, const char *msg) { return fail(code, "%s", msg); }
__attribute__((visibility("hidden"))) int ktb_internal_sms(const ktb_oligo *h) { return h->sm_count; }
__attribute__((visibility("hidden"))) uint64_t ktb_internal_launches(const ktb_oligo *h) { return h->stats.launches; }

namespace {

int check_args(const ktb_oligo *h, int canonical, int norm_mode, int out_dtype) {
    if (!h) return fail(KTB_ERR_ARG, "null handle");
    if (canonical != 0 && canonical != 1) return fail(KTB_ERR_ARG, "canonical must be 0 or 1");
    if (norm_mode < 0 || norm_mode > 2) return fail(KTB_ERR_ARG, "unknown norm_mode %d", norm_mode);
    if (out_dtype < 0 || out_dtype > 2) return fail(KTB_ERR_ARG, "unknown out_dtype %d", out_dtype);
    if (out_dtype == KTB_OUT_U32 && norm_mode != KTB_NORM_COUNTS)
        return fail(KTB_ERR_ARG, "KTB_OUT_U32 requires KTB_NORM_COUNTS");
    return KTB_OK;
}

__global__ void rebase_offsets_kernel(uint64_t *offs, uint64_t count, uint64_t bias) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count;
         i += (uint64_t)gridDim.x * blockDim.x)
        offs[i] -= bias;
}

double now_ms() {
    using namespace std::chrono;
    return duration<double, std::milli>(steady_clock::now().time_since_epoch()).count();
}

// Copies a table into a new device allocation of exactly its size.
cudaError_t upload(uint32_t **d, const std::vector<uint32_t> &tab) {
    const cudaError_t e = cudaMalloc(d, tab.size() * 4);
    return e != cudaSuccess ? e : cudaMemcpy(*d, tab.data(), tab.size() * 4, cudaMemcpyHostToDevice);
}

}  // namespace

// =================================================================================================
extern "C" {

const char *ktb_last_error(void) { return g_err.c_str(); }
int ktb_abi_version(void) { return KTB_ABI_VERSION; }

int ktb_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

int ktb_oligo_create(int k, int device, ktb_oligo **out) {
    if (!out) return fail(KTB_ERR_ARG, "out is NULL");
    *out = nullptr;
    if (k < 1 || k > KTB_MAX_K) return fail(KTB_ERR_ARG, "k must be in 1..%d (got %d)", KTB_MAX_K, k);
    const int ndev = ktb_device_count();
    if (ndev <= 0) return fail(KTB_ERR_NODEVICE, "no CUDA device available (this library has no CPU path)");
    if (device < 0 || device >= ndev) return fail(KTB_ERR_ARG, "device %d out of range (0..%d)", device, ndev - 1);

    ktb_oligo *h = new ktb_oligo();
    h->k = k;
    h->device = device;
    h->ncodes = 1ULL << (2 * k);
    // kmer_pos_maps (kmer/src/kmer.rs:54-73): canonical codes in ascending order get ranks 0..count-1.
    // Walking x upward and keeping x when x <= rc(x) visits exactly the sorted canonical set.
    h->rank_of_canon.assign(h->ncodes, 0);
    std::vector<uint32_t> rank_full(h->ncodes);
    for (uint64_t x = 0; x < h->ncodes; ++x) {
        if (x <= rev_comp(x, k)) {
            h->rank_of_canon[x] = (uint32_t)h->canon_of_rank.size();
            h->canon_of_rank.push_back((uint32_t)x);
        }
    }
    h->dim_canon = h->canon_of_rank.size();
    for (uint64_t x = 0; x < h->ncodes; ++x) {
        const uint64_t rc = rev_comp(x, k);
        rank_full[x] = h->rank_of_canon[x < rc ? x : rc];
    }

    auto bail = [&](int rc) {
        ktb_oligo_destroy(h);
        return rc;
    };
    DeviceGuard device_guard_(device);
    if (device_guard_.err != cudaSuccess) return bail(fail(KTB_ERR_CUDA, "cudaSetDevice(%d) failed", device));
    cudaDeviceProp prop{};
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess)
        return bail(fail(KTB_ERR_CUDA, "cudaGetDeviceProperties failed"));
    h->sm_count = prop.multiProcessorCount;
    h->smem_optin = prop.sharedMemPerBlockOptin;
    h->coop_launch = prop.cooperativeLaunch != 0;   // wave_kernel needs co-resident CTAs; else the multi-launch variant

#define CUB(call)                                                                                  \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess)                                                                     \
            return bail(fail(KTB_ERR_CUDA, "%s failed: %s", #call, cudaGetErrorString(e_)));       \
    } while (0)

    CUB(upload(&h->d_rank_full, rank_full));
    std::vector<uint32_t> cor(h->canon_of_rank);
    while (cor.size() % 4) cor.push_back(0);
    CUB(upload(&h->d_canon_of_rank, cor));
    {
        std::vector<uint32_t> perm(cor.size(), 0);
        const uint64_t nblk = h->dim_canon / 128;
        for (uint64_t b = 0; b < nblk; ++b)
            for (uint32_t l = 0; l < 32; ++l)
                for (uint32_t e = 0; e < 4; ++e) perm[b * 128 + 4 * l + e] = cor[b * 128 + 32 * e + l];
        CUB(upload(&h->d_canon_perm, perm));
        if (!(k & 1) && k >= 6 && k <= 8) {  // rank tables of seq_kernel mode 7 (see kernels.cuh)
            const uint32_t hd = k / 2, H = 1u << (2 * hd), wpr = H / 32;   // halves of hd bases, words per row
            std::vector<uint32_t> tab((size_t)H * wpr + ((size_t)H * wpr + 1) / 2, 0);
            uint16_t *pref = reinterpret_cast<uint16_t *>(tab.data() + (size_t)H * wpr);
            uint32_t running = 0;
            for (uint32_t a = 0; a < H; ++a) {
                for (uint32_t w = 0; w < wpr; ++w) {
                    uint32_t bits = 0;
                    for (uint32_t i = 0; i < 32; ++i)
                        if ((uint32_t)rev_comp(32 * w + i, hd) >= a) bits |= 1u << i;   // (a, R) canonical <=> a <= rc(R)
                    tab[(size_t)a * wpr + w] = bits;
                    pref[(size_t)a * wpr + w] = (uint16_t)running;
                    running += (uint32_t)__builtin_popcount(bits);
                }
            }
            if (running == h->dim_canon && h->dim_canon <= 65535u + 32u) {
                h->even_words = H * wpr;
                CUB(upload(&h->d_even_tab, tab));
            }
        }
        if (k & 1) {  // dense half-size index of seq_kernel mode 4 (see kernels.cuh)
            const uint32_t midbit = 1u << (2 * (k / 2) + 1);
            std::vector<uint32_t> mb(cor.size(), 0), mbp(cor.size(), 0);
            for (uint64_t j = 0; j < h->dim_canon; ++j) {
                const uint32_t c = cor[j];
                const uint32_t sel = (c & midbit) ? (uint32_t)rev_comp(c, k) : c;
                const uint32_t d = (sel & (midbit - 1)) | ((sel >> 1) & ~(midbit - 1));
                const uint32_t m = 2 * (k / 2) + 1;                 // bit index of midbit
                const uint32_t skew = (uint32_t)((4ull << m) >> 9); // words of skew per row, as in the kernel
                mb[j] = d + (d >> m) * skew;
                h->mb_entries = std::max<uint64_t>(h->mb_entries, (uint64_t)mb[j] + 1);
            }
            for (uint64_t b = 0; b < nblk; ++b)
                for (uint32_t l = 0; l < 32; ++l)
                    for (uint32_t e = 0; e < 4; ++e) mbp[b * 128 + 4 * l + e] = mb[b * 128 + 32 * e + l];
            CUB(upload(&h->d_mb_of_rank, mb));
            CUB(upload(&h->d_mb_perm, mbp));
        }
    }
    if (k == 7) {   // long_kernel MODE_K7: bin of a class = [b3 b4 b5 b6 | b0 b1 b2] of the strand whose middle base is A/C
        std::vector<uint32_t> word(h->dim_canon);
        for (uint64_t j = 0; j < h->dim_canon; ++j) {
            uint32_t sgl = h->canon_of_rank[j];
            if (((sgl >> 6) & 3u) >= 2u) sgl = (uint32_t)rev_comp(sgl, 7);
            word[j] = ((sgl & 0xFFu) << 6) | ((sgl >> 8) & 0x3Fu);
        }
        const std::vector<uint32_t> order = conflict_free_groups(word);
        if (!order.empty()) {
            // warp iteration w, lane l, element q  <-  group 4w + q, lane l   (one 128-bit load per lane and iteration)
            std::vector<uint32_t> sched(h->dim_canon);
            for (uint64_t g = 0; g < h->dim_canon / 32; ++g)
                for (uint32_t l = 0; l < 32; ++l) {
                    const uint32_t j = order[g * 32 + l];
                    sched[((g >> 2) * 32 + l) * 4 + (g & 3)] = (word[j] * 4u) | ((j * 4u) << 16);
                }
            CUB(upload(&h->d_k7_sched, sched));
        }
    }
    // long_kernel MODE_FWD: fold table, rank -> (c, rc(c)).  k = 6 stays with seq_kernel: its fold gathers hist[rc(c)] for
    // consecutive c, which differ in their TOP digits, i.e. 32 lanes in one bank (measured 2x slower, profiles/r2_sweeps.txt)
    if (k >= 3 && k <= 5 && (h->dim_canon % 4) == 0) {
        std::vector<uint32_t> sched(h->dim_canon);
        for (uint64_t j = 0; j < h->dim_canon; ++j) {
            const uint32_t c = h->canon_of_rank[j], r = (uint32_t)rev_comp(c, k);
            sched[j] = (c * 4u) | (((r == c) ? (uint32_t)h->ncodes : r) * 4u) << 16;
        }
        CUB(upload(&h->d_fwd_sched, sched));
    }
    {   // bitmap of the canonical codes + running rank per pair of words: rank(c) = prefix[w / 2] + popc(bits below c).
        // wave_kernel<2> keeps the whole table in shared memory (k <= 10); count_kernel loads one segment's slice.
        const uint64_t words = h->ncodes / 32;
        const uint64_t bytes = words * 4 + (words / 2) * 4;
        if (h->ncodes >= 64 && h->dim_canon * 4 > 64 * 1024) {
            std::vector<uint32_t> tab(words + words / 2, 0);
            uint32_t running = 0;
            bool aligned = true;
            for (uint64_t w = 0; w < words; ++w) {
                if (!(w & 1)) tab[words + w / 2] = running;
                if ((w & 255) == 0 && (running & 3)) aligned = false;   // segment boundaries (2^13 codes and coarser)
                uint32_t bits = 0;
                for (uint32_t i = 0; i < 32; ++i) {
                    const uint64_t x = 32 * w + i;
                    if (x <= rev_comp(x, k)) bits |= 1u << i;
                }
                tab[w] = bits;
                running += (uint32_t)__builtin_popcount(bits);
            }
            h->wave_tab_words = (uint32_t)words;
            h->wave_tab_in_smem = bytes + 4096 <= h->smem_optin;
            h->wave_seg_aligned = aligned;
            CUB(upload(&h->d_wave_tab, tab));
        }
    }
    if (h->ncodes <= (uint64_t)ktb::SHORT_MAX_CODES) {
        std::vector<uint32_t> tc(h->ncodes), tr(h->ncodes);
        for (uint64_t x = 0; x < h->ncodes; ++x) {
            const uint32_t a = rank_full[x], b = (uint32_t)x;
            tc[x] = ((a & ~3u) << 22) | ((a & 3u) * 8u);
            tr[x] = ((b & ~3u) << 22) | ((b & 3u) * 8u);
        }
        CUB(upload(&h->d_short_tab_canon, tc));
        CUB(upload(&h->d_short_tab_raw, tr));
    }
    CUB(cudaMalloc(&h->d_counters, 16 * sizeof(unsigned long long)));
    for (auto &s : h->sets) {
        CUB(cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking));
        for (auto &e : s.ev) CUB(cudaEventCreate(&e));
    }
    for (auto &a : h->aux) CUB(cudaStreamCreateWithFlags(&a, cudaStreamNonBlocking));
    for (auto &e : h->aux_ev) CUB(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    CUB(cudaEventCreate(&h->ref_ev));
    // cudaMemcpy from pageable memory may return while the DMA to the device is still in flight, and the
    // handle's non-blocking streams do not order against the default stream: make the tables visible now.
    CUB(cudaDeviceSynchronize());
#undef CUB
    *out = h;
    return KTB_OK;
}

void ktb_oligo_destroy(ktb_oligo *h) {
    if (!h) return;
    DeviceGuard device_guard_(h->device);
    for (auto &s : h->sets) {
        if (s.stream) {
            cudaStreamSynchronize(s.stream);
            cudaStreamDestroy(s.stream);
        }
        for (auto &e : s.ev)
            if (e) cudaEventDestroy(e);
    }
    for (auto &a : h->aux) if (a) { cudaStreamSynchronize(a); cudaStreamDestroy(a); }
    for (auto &e : h->aux_ev) if (e) cudaEventDestroy(e);
    if (h->ref_ev) cudaEventDestroy(h->ref_ev);
    for (auto &e : h->wave_ev) if (e) cudaEventDestroy(e);
    for (uint32_t *t : {h->d_rank_full, h->d_canon_of_rank, h->d_canon_perm, h->d_mb_of_rank, h->d_mb_perm, h->d_even_tab,
                        h->d_wave_tab, h->d_k7_sched, h->d_fwd_sched, h->d_short_tab_canon, h->d_short_tab_raw})
        if (t) cudaFree(t);
    if (h->d_counters) cudaFree(h->d_counters);
    delete h;   // the scratch buffers free themselves, on this device
}

int ktb_oligo_k(const ktb_oligo *h) { return h ? h->k : 0; }

uint64_t ktb_oligo_dim(const ktb_oligo *h, int canonical) {
    if (!h) return 0;
    return canonical ? h->dim_canon : h->ncodes;
}

int ktb_oligo_header(const ktb_oligo *h, int canonical, char *buf, size_t cap) {
    if (!h || !buf) return fail(KTB_ERR_ARG, "null argument");
    const uint64_t dim = ktb_oligo_dim(h, canonical);
    if (cap < dim * (uint64_t)h->k) return fail(KTB_ERR_ARG, "header buffer too small (%zu < %llu)", cap,
                                               (unsigned long long)(dim * h->k));
    static const char L[4] = {'A', 'C', 'G', 'T'};
    for (uint64_t j = 0; j < dim; ++j) {  // numeric_to_kmer, kmer/src/lib.rs:19-34
        uint64_t code = canonical ? h->canon_of_rank[j] : j;
        for (int i = h->k - 1; i >= 0; --i) {
            buf[j * h->k + i] = L[code & 3];
            code >>= 2;
        }
    }
    return KTB_OK;
}

int ktb_oligo_pos_maps(const ktb_oligo *h, uint64_t *pos_map, uint64_t *pos_to_kmer, uint64_t *count) {
    if (!h) return fail(KTB_ERR_ARG, "null handle");
    if (pos_map)
        for (uint64_t x = 0; x < h->ncodes; ++x) pos_map[x] = h->rank_of_canon[x];
    if (pos_to_kmer)
        for (uint64_t j = 0; j < h->dim_canon; ++j) pos_to_kmer[j] = h->canon_of_rank[j];
    if (count) *count = h->dim_canon;
    return KTB_OK;
}

int ktb_oligo_set_option(ktb_oligo *h, const char *key, int64_t value) {
    if (!h || !key) return fail(KTB_ERR_ARG, "null argument");
    if (!strcmp(key, "chunk_bytes")) {
        if (value < (1 << 16)) return fail(KTB_ERR_ARG, "chunk_bytes too small");
        h->chunk_bytes = value;
    } else if (!strcmp(key, "force_path")) {
        h->force_path = (int)value;
    } else if (!strcmp(key, "long_warps")) {
        if (value != 0 && value != 4 && value != 8 && value != 10) return fail(KTB_ERR_ARG, "long_warps must be 0, 4, 8 or 10");
        h->long_warps = (int)value;
    } else if (!strcmp(key, "k7_mid")) {
        h->k7_mid = (int)value;
    } else if (!strcmp(key, "fwd_replicas")) {
        h->fwd_replicas = (int)value;
    } else if (!strcmp(key, "fwd_fold")) {
        h->fwd_fold = (int)value;
    } else if (!strcmp(key, "fwd_min_len")) {
        h->fwd_min_len = value;
    } else if (!strcmp(key, "bucket")) {
        h->bucket = (int)value;
    } else if (!strcmp(key, "k8_long")) {
        if (value < 0 || value > 1) return fail(KTB_ERR_ARG, "k8_long must be 0 or 1");
        h->k8_long = (int)value;
    } else if (!strcmp(key, "longest_first")) {
        if (value < 0 || value > 1) return fail(KTB_ERR_ARG, "longest_first must be 0 or 1");
        h->longest_first = (int)value;
    } else if (!strcmp(key, "bucket_hist_kb")) {
        if (value != 64 && value != 96) return fail(KTB_ERR_ARG, "bucket_hist_kb must be 64 or 96");
        h->bucket_hist_kb = (int)value;
    } else if (!strcmp(key, "bucket_wave_ctas")) {
        if (value < 1 || value > 4) return fail(KTB_ERR_ARG, "bucket_wave_ctas must be in 1..4");
        h->bucket_wave_ctas = (int)value;
    } else if (!strcmp(key, "bucket_waves")) {
        if (value < 1 || value > 64) return fail(KTB_ERR_ARG, "bucket_waves must be in 1..64");
        h->bucket_waves = (int)value;
    } else if (!strcmp(key, "bucket_log2_seg")) {
        if (value < 13 || value > 14) return fail(KTB_ERR_ARG, "bucket_log2_seg must be 13 or 14");
        h->bucket_log2_seg = (int)value;
    } else if (!strcmp(key, "packed16")) {
        h->packed16 = (int)value;
    } else if (!strcmp(key, "even_rank")) {
        h->even_rank = (int)value;
    } else if (!strcmp(key, "dense_odd")) {
        h->dense_odd = (int)value;
    } else if (!strcmp(key, "global_steps_per_warp")) {
        h->global_steps_per_warp = (int)value;
    } else if (!strcmp(key, "wave_persistent")) {
        h->wave_persistent = value != 0;
    } else if (!strcmp(key, "seq_grab")) {
        if (value < 0 || value > 1024) return fail(KTB_ERR_ARG, "seq_grab must be in 0..1024");
        h->seq_grab = (int)value;
    } else if (!strcmp(key, "wave_smem_rank")) {
        h->wave_smem_rank = value != 0;
    } else if (!strcmp(key, "wave_budget_bytes")) {
        if (value < 1) return fail(KTB_ERR_ARG, "wave_budget_bytes must be positive");
        h->wave_budget_bytes = value;
    } else if (!strcmp(key, "global_wave_bytes")) {
        if (value < 1) return fail(KTB_ERR_ARG, "global_wave_bytes must be positive");
        h->global_wave_bytes = value;
    } else if (!strcmp(key, "seq_threads")) {
        if (value != 0 && (value < 32 || value > 1024 || value % 32)) return fail(KTB_ERR_ARG, "seq_threads must be a multiple of 32 in 32..1024");
        h->seq_threads = (int)value;
    } else {
        return fail(KTB_ERR_ARG, "unknown option '%s'", key);
    }
    return KTB_OK;
}

int ktb_oligo_last_stats(const ktb_oligo *h, ktb_stats *out) {
    if (!h || !out) return fail(KTB_ERR_ARG, "null argument");
    *out = h->stats;
    return KTB_OK;
}

int ktb_oligo_vectorise_device(ktb_oligo *h, const uint8_t *d_bases, const uint64_t *d_offsets, uint64_t n,
                               uint64_t total_bases, int canonical, int norm_mode, int out_dtype,
                               void *d_out, uint64_t *d_totals, void *stream) {
    if (int rc = check_args(h, canonical, norm_mode, out_dtype)) return rc;
    if (n && (!d_offsets || !d_out)) return fail(KTB_ERR_ARG, "null device pointer");
    if (total_bases && !d_bases) return fail(KTB_ERR_ARG, "null bases pointer");
    if (((uintptr_t)d_bases & 15) || ((uintptr_t)d_out & 15))
        return fail(KTB_ERR_ARG, "d_bases and d_out must be 16-byte aligned");
    ON_DEVICE(h->device);
    h->stats = ktb_stats{};
    return dispatch_device(h, d_bases, d_offsets, n, total_bases, canonical, norm_mode, out_dtype, d_out,
                           d_totals, (cudaStream_t)stream);
}

int ktb_oligo_vectorise(ktb_oligo *h, const uint8_t *bases, const uint64_t *offsets, uint64_t n, int canonical,
                        int norm_mode, int out_dtype, void *out, uint64_t *totals) {
    if (int rc = check_args(h, canonical, norm_mode, out_dtype)) return rc;
    if (n && (!offsets || !out)) return fail(KTB_ERR_ARG, "null pointer");
    ON_DEVICE(h->device);
    const double t0 = now_ms();
    h->stats = ktb_stats{};
    if (n == 0) return KTB_OK;
    if (offsets[n] > offsets[0] && !bases) return fail(KTB_ERR_ARG, "null bases pointer");
    // The offsets are validated chunk by chunk, right before a chunk is queued: reading 8 bytes per sequence on one
    // host thread (10 ms for the 10 M reads of the headline config) then runs under the copies of the chunks before it
    // instead of in front of the whole call.  A chunk's extent must also stay inside [offsets[0], offsets[n]].
    if (offsets[n] < offsets[0]) return fail(KTB_ERR_ARG, "offsets must be non-decreasing (last < first)");

    const uint64_t dim = ktb_oligo_dim(h, canonical);
    const size_t esize = out_dtype == KTB_OUT_F64 ? 8 : 4;
    const uint64_t row_bytes = dim * esize;
    uint64_t rows_per_chunk = std::max<uint64_t>(1, (uint64_t)h->chunk_bytes / row_bytes);
    const uint64_t max_chunk_bases = 1ull << 30;

    bool has[NBUF] = {false, false, false};
    // h2d_ms / kernel_ms / d2h_ms are the time during which AT LEAST ONE copy (kernel) of that kind was running: the
    // three stream sets overlap, so per-chunk durations are kept as intervals on one clock (an event recorded at the
    // start of the call) and merged at the end — their plain sum would exceed the wall time.
    struct Span { float a, b; };
    std::vector<Span> spans[3];
    CU(cudaEventRecord(h->ref_ev, h->sets[0].stream));
    auto drain = [&](int b) -> int {
        ChunkSet &s = h->sets[b];
        if (!has[b]) return KTB_OK;
        CU(cudaStreamSynchronize(s.stream));
        const int first[3] = {0, 4, 2}, last[3] = {1, 2, 3};
        for (int q = 0; q < 3; ++q) {
            Span sp{};
            CU(cudaEventElapsedTime(&sp.a, h->ref_ev, s.ev[first[q]]));
            CU(cudaEventElapsedTime(&sp.b, h->ref_ev, s.ev[last[q]]));
            spans[q].push_back(sp);
        }
        has[b] = false;
        return KTB_OK;
    };
    auto union_ms = [](std::vector<Span> &v) -> double {
        std::sort(v.begin(), v.end(), [](const Span &x, const Span &y) { return x.a < y.a; });
        double total = 0;
        float cur_a = 0, cur_b = -1;
        for (const Span &sp : v) {
            if (cur_b < cur_a || sp.a > cur_b) {
                if (cur_b >= cur_a) total += cur_b - cur_a;
                cur_a = sp.a; cur_b = sp.b;
            } else if (sp.b > cur_b) {
                cur_b = sp.b;
            }
        }
        if (cur_b >= cur_a) total += cur_b - cur_a;
        return total;
    };

    int b = 0;
    cudaEvent_t prev_kernels_done = nullptr;
    uint64_t total_launches = 0;
    uint64_t checked = 0;   // offsets[0 .. checked] are known to be non-decreasing and <= offsets[n]
    auto bad_offsets = [&](uint64_t upto) -> int64_t {
        for (; checked < upto; ++checked)
            if (offsets[checked + 1] < offsets[checked] || offsets[checked + 1] > offsets[n]) return (int64_t)checked;
        return -1;
    };
    for (uint64_t i0 = 0; i0 < n;) {
        uint64_t i1 = std::min(n, i0 + rows_per_chunk);
        if (const int64_t bad = bad_offsets(i1); bad >= 0) {
            for (int q = 0; q < NBUF; ++q) drain(q);   // nothing of this call may still be writing into `out`
            return fail(KTB_ERR_ARG, "offsets must be non-decreasing (at %llu)", (unsigned long long)bad);
        }
        // cap the bases per chunk (always keep at least one sequence)
        if (offsets[i1] - offsets[i0] > max_chunk_bases && i1 > i0 + 1) {
            const uint64_t *lo = offsets + i0 + 1, *hi = offsets + i1;
            const uint64_t *it = std::upper_bound(lo, hi, offsets[i0] + max_chunk_bases);
            i1 = std::max<uint64_t>(i0 + 1, (uint64_t)(it - offsets) - 1);
        }
        const uint64_t cn = i1 - i0;
        const uint64_t b0 = offsets[i0] & ~15ull;  // keep the 16-byte phase of the caller's buffer
        const uint64_t nb = offsets[i1] - b0;
        ChunkSet &s = h->sets[b];
        if (int rc = drain(b)) return rc;
        if (int rc = s.bases.ensure(nb + 64)) return rc;
        if (int rc = s.offsets.ensure((cn + 1) * 8)) return rc;
        if (int rc = s.out.ensure(cn * row_bytes)) return rc;
        if (totals)
            if (int rc = s.totals.ensure(cn * 8)) return rc;
        CU(cudaEventRecord(s.ev[0], s.stream));
        if (nb) CU(cudaMemcpyAsync(s.bases.p, bases + b0, nb, cudaMemcpyHostToDevice, s.stream));
        CU(cudaMemcpyAsync(s.offsets.p, offsets + i0, (cn + 1) * 8, cudaMemcpyHostToDevice, s.stream));
        CU(cudaEventRecord(s.ev[1], s.stream));
        if (b0) {
            rebase_offsets_kernel<<<(unsigned)std::min<uint64_t>((cn + 256) / 256, 1024), 256, 0, s.stream>>>(
                (uint64_t *)s.offsets.p, cn + 1, b0);
            CU(cudaGetLastError());
            total_launches++;
        }
        // The work counters, reject lists and scratch rows live in the handle, not in the chunk set: the
        // kernels of consecutive chunks must not overlap (copies still do).  Chain them with an event.
        if (prev_kernels_done) CU(cudaStreamWaitEvent(s.stream, prev_kernels_done, 0));
        CU(cudaEventRecord(s.ev[4], s.stream));
        const ktb_stats keep = h->stats;
        if (int rc = dispatch_device(h, (const uint8_t *)s.bases.p, (const uint64_t *)s.offsets.p, cn, nb,
                                     canonical, norm_mode, out_dtype, s.out.p,
                                     totals ? (uint64_t *)s.totals.p : nullptr, s.stream))
            return rc;
        total_launches += h->stats.launches - keep.launches;
        CU(cudaEventRecord(s.ev[2], s.stream));
        prev_kernels_done = s.ev[2];
        CU(cudaMemcpyAsync((uint8_t *)out + i0 * row_bytes, s.out.p, cn * row_bytes, cudaMemcpyDeviceToHost,
                           s.stream));
        if (totals) CU(cudaMemcpyAsync(totals + i0, s.totals.p, cn * 8, cudaMemcpyDeviceToHost, s.stream));
        CU(cudaEventRecord(s.ev[3], s.stream));
        h->stats.h2d_bytes += nb + (cn + 1) * 8;
        h->stats.d2h_bytes += cn * row_bytes + (totals ? cn * 8 : 0);
        has[b] = true;
        b = (b + 1) % NBUF;
        i0 = i1;
    }
    for (int q = 0; q < NBUF; ++q)
        if (int rc = drain(q)) return rc;
    h->stats.h2d_ms = union_ms(spans[0]);
    h->stats.kernel_ms = union_ms(spans[1]);
    h->stats.d2h_ms = union_ms(spans[2]);
    h->stats.launches = total_launches;
    h->stats.wall_ms = now_ms() - t0;
    return KTB_OK;
}

void *ktb_host_alloc(size_t bytes) {
    void *p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocPortable) != cudaSuccess) {
        fail(KTB_ERR_NOMEM, "cudaHostAlloc(%zu) failed: %s", bytes, cudaGetErrorString(cudaGetLastError()));
        return nullptr;
    }
    ktb_internal_register_host(p, bytes);
    return p;
}

void ktb_host_free(void *p) {
    if (p) ktb_internal_free_host(p);
}

int ktb_debug_nt4_table(ktb_oligo *h, uint8_t *out256) {
    if (!h || !out256) return fail(KTB_ERR_ARG, "null argument");
    ON_DEVICE(h->device);
    uint8_t *d = nullptr;
    CU(cudaMalloc(&d, 256));
    ktb::nt4_table_kernel<<<1, 256>>>(d);
    cudaError_t e = cudaMemcpy(out256, d, 256, cudaMemcpyDeviceToHost);
    cudaFree(d);
    if (e != cudaSuccess) return fail(KTB_ERR_CUDA, "nt4 table copy failed: %s", cudaGetErrorString(e));
    return KTB_OK;
}

}  // extern "C"
