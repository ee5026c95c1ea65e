// file_api.cu — file-level driver behind `kmertools comp oligo` (see include/kmertools_b200.h).
// Host side: streaming FASTA/FASTQ parse into pinned, offset-indexed buffers; two buffer sets so that
// parsing batch b+1 overlaps the GPU work and the D2H copy of batch b; finished batches go to an ordered
// asynchronous writer (span_writer.h: `-t` threads copy disjoint spans into a shared mapping of the output, as the
// reference's mmap writer does), so writing batch b also overlaps batch b+1.  Device side: counts + format_norm_kernel.
#include "../../include/kmertools_b200.h"
#include "device_guard.h"
#include "fastx.h"
#include "span_writer.h"
#include "textfmt.cuh"

#include <atomic>
#include <charconv>
#include <sys/stat.h>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <filesystem>
#include <mutex>
#include <string>
#include <sched.h>
#include <thread>
#include <vector>

int ktb_internal_dispatch(ktb_oligo *h, const uint8_t *d_bases, const uint64_t *d_offsets, uint64_t n,
                          uint64_t total_bases, int canonical, int norm_mode, int out_dtype, void *d_out,
                          uint64_t *d_totals, cudaStream_t st);
int ktb_internal_fail(int code, const char *msg);
int ktb_internal_sms(const ktb_oligo *h);
uint64_t ktb_internal_launches(const ktb_oligo *h);
void ktb_internal_counter_table(const ktb_counter *c, const uint64_t **keys, const uint64_t **counts);
int ktb_internal_coverage_args(uint32_t bin_size, uint32_t bin_count, int norm_mode, int out_dtype);

namespace {

double now_ms() {
    using namespace std::chrono;
    return duration<double, std::milli>(steady_clock::now().time_since_epoch()).count();
}

struct Pinned {
    void *p = nullptr;
    size_t cap = 0;
    bool ensure(size_t bytes) {
        if (bytes <= cap) return true;
        void *q = nullptr;
        if (cudaHostAlloc(&q, bytes, cudaHostAllocDefault) != cudaSuccess) return false;
        if (p) cudaFreeHost(p);
        p = q;
        cap = bytes;
        return true;
    }
    bool grow_keep(size_t bytes, size_t keep) {  // enlarge, preserving the first `keep` bytes
        if (bytes <= cap) return true;
        void *q = nullptr;
        if (cudaHostAlloc(&q, bytes, cudaHostAllocDefault) != cudaSuccess) return false;
        if (p && keep) memcpy(q, p, keep);
        if (p) cudaFreeHost(p);
        p = q;
        cap = bytes;
        return true;
    }
    ~Pinned() { if (p) cudaFreeHost(p); }
};

struct Dev {
    void *p = nullptr;
    size_t cap = 0;
    bool ensure(size_t bytes) {
        if (bytes <= cap) return true;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        if (cudaMalloc(&p, bytes + bytes / 8 + 256) != cudaSuccess) { p = nullptr; return false; }
        cap = bytes + bytes / 8 + 256;
        return true;
    }
    ~Dev() { if (p) cudaFree(p); }
};

// Host-formatted text.  resize() leaves new bytes uninitialised: a part sized for the longest text its rows can have
// touches (and keeps resident) only the pages the text is written to.
template <class T>
struct NoInitAlloc : std::allocator<T> {
    template <class U> struct rebind { using other = NoInitAlloc<U>; };
    NoInitAlloc() = default;
    template <class U> NoInitAlloc(const NoInitAlloc<U> &) noexcept {}
    template <class U> void construct(U *p) noexcept { ::new ((void *)p) U; }
    template <class U, class... A> void construct(U *p, A &&...a) { ::new ((void *)p) U(std::forward<A>(a)...); }
};
using Text = std::vector<char, NoInitAlloc<char>>;

struct Set {
    Pinned h_bases, h_offsets, h_out;
    Dev d_bases, d_offsets, d_counts, d_totals, d_text;
    cudaStream_t stream = nullptr;
    cudaEvent_t kernels_done = nullptr;
    uint64_t n = 0, nbases = 0, out_bytes = 0;
    bool pending = false;
    bool writing = false;                      // rows handed to the writer, buffers not reusable yet
    ktb::SpanWriter::Ticket ticket;
    std::vector<Text> parts;                   // host-formatted text (counts / CGR), one part per formatting thread
    ~Set() {
        if (kernels_done) cudaEventDestroy(kernels_done);
        if (stream) cudaStreamDestroy(stream);
    }
};

// The two buffer sets of the last run are kept for the next one on the same device: page-locking costs ~0.5 ms
// per MB (several times that right after a large pinned region was released), which was half of a warm 1 GB run.
// One cached pair per process, handed to one caller at a time; never destroyed at exit (the CUDA runtime may be
// gone by then), ktb_release_cached_buffers() frees it on request.
struct SetPair {
    Set sets[2];
    int device = -1;
};
std::mutex g_pool_mutex;
SetPair *g_pool = nullptr;

SetPair *acquire_sets(int device) {
    SetPair *sp = nullptr;
    {
        std::lock_guard<std::mutex> lk(g_pool_mutex);
        if (g_pool && g_pool->device == device) {
            sp = g_pool;
            g_pool = nullptr;
        }
    }
    if (!sp) {
        sp = new SetPair();
        sp->device = device;
    }
    for (auto &s : sp->sets) {
        s.n = s.nbases = s.out_bytes = 0;
        s.pending = false;
        s.writing = false;
        s.ticket = ktb::SpanWriter::Ticket();
        if ((!s.stream && cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking) != cudaSuccess) ||
            (!s.kernels_done && cudaEventCreateWithFlags(&s.kernels_done, cudaEventDisableTiming) != cudaSuccess)) {
            delete sp;
            return nullptr;
        }
    }
    return sp;
}

void release_sets(SetPair *sp) {
    if (!sp) return;
    for (auto &s : sp->sets)
        if (s.stream) cudaStreamSynchronize(s.stream);   // an error path may leave copies in flight
    SetPair *old = nullptr;
    {
        std::lock_guard<std::mutex> lk(g_pool_mutex);
        old = g_pool;
        g_pool = sp;
    }
    delete old;
}

// `-t` (kmertools/src/args.rs:249-251; 0 = all cores): threads of the output writer and of the host formatter
// (all cores = the CPUs this process may run on, at most 8: sixteen writer threads measured no faster on tmpfs —
// 149 against 145 ms per GB, profiles/r2_cli_writer.txt — and write() on a disk file system uses one anyway)
int host_threads(int threads) {
    int hw = (int)std::max(1u, std::thread::hardware_concurrency());
    cpu_set_t set;
    CPU_ZERO(&set);
    if (sched_getaffinity(0, sizeof(set), &set) == 0 && CPU_COUNT(&set) > 0) hw = CPU_COUNT(&set);
    return threads > 0 ? std::min(threads, 64) : std::min(hw, 8);
}

// Bases per input batch: 32 MB, less for a small regular file (which should not page-lock 32 MB per buffer).
size_t input_bases_cap(const std::string &in) {
    size_t cap = 32u << 20;
    struct stat sb;
    if (in != "-" && stat(in.c_str(), &sb) == 0 && S_ISREG(sb.st_mode)) {
        const bool gz = in.size() > 3 && in.compare(in.size() - 3, 3, ".gz") == 0;
        const size_t est = (size_t)sb.st_size * (gz ? 8 : 1) + (1u << 20);
        if (est < cap) cap = est;
    }
    return cap;
}

// Fills `bases` with the next batch of records (offs: its n + 1 offsets), growing the buffer and *cap when one record
// does not fit.
int fill_batch(ktb::FastxParser &parser, Pinned &bases, size_t *cap, size_t max_records, size_t *used,
               std::vector<uint64_t> *offs) {
    offs->assign(1, 0);
    *used = 0;
    for (;;) {
        const long got = parser.fill((uint8_t *)bases.p, bases.cap, used, offs, max_records);
        if (got < 0) return ktb_internal_fail(KTB_ERR_IO, parser.error().c_str());
        if (got == 0 && parser.need_bytes() && *used == 0) {  // one record larger than the buffer
            *cap = parser.need_bytes() + (parser.need_bytes() >> 2) + 4096;
            if (!bases.grow_keep(*cap, 0)) return ktb_internal_fail(KTB_ERR_NOMEM, "pinned allocation failed");
            continue;
        }
        return KTB_OK;
    }
}

// Opens a sequence input of the counting drivers: "-" (stdin) sniffs the first byte, a path's extension decides.
int open_seq_input(const std::string &path, ktb::ByteSource *src, ktb::SeqFormat *fmt) {
    std::string err;
    if (!src->open(path, &err)) return ktb_internal_fail(KTB_ERR_IO, err.c_str());
    if (path == "-") *fmt = (src->peek_first_byte() == '>') ? ktb::SeqFormat::Fasta : ktb::SeqFormat::Fastq;
    else if (!ktb::format_from_path(path, fmt))
        return ktb_internal_fail(KTB_ERR_IO, "unknown sequence file extension (expected .fa/.fasta/.fna/.fq/.fastq[.gz])");
    return KTB_OK;
}

// Counts every record of `parser` into c: batch b is added on a worker thread while the caller parses batch b + 1 into
// the other buffer.  Adds the records, bases, parse time and the time spent waiting for adds to *st.
int count_into(ktb_counter *c, ktb::FastxParser &parser, size_t bases_cap, ktb_file_stats *st) {
    Pinned hbases[2];
    std::vector<uint64_t> offs[2];
    const size_t max_records = 4u << 20;
    std::thread adder;
    int add_rc = KTB_OK;
    std::string add_err;
    auto join = [&]() -> int {
        if (!adder.joinable()) return KTB_OK;
        const double t0 = now_ms();
        adder.join();
        st->gpu_wait_ms += now_ms() - t0;
        return add_rc ? ktb_internal_fail(add_rc, add_err.c_str()) : KTB_OK;
    };
    struct JoinGuard { std::thread *t; ~JoinGuard() { if (t->joinable()) t->join(); } } join_guard{&adder};
    for (int b = 0;; ++b) {
        Pinned &hb = hbases[b & 1];
        std::vector<uint64_t> &of = offs[b & 1];
        const double tp0 = now_ms();
        if (!hb.ensure(bases_cap)) return ktb_internal_fail(KTB_ERR_NOMEM, "pinned allocation failed");
        size_t used = 0;
        if (int rc = fill_batch(parser, hb, &bases_cap, max_records, &used, &of)) return rc;
        st->parse_ms += now_ms() - tp0;
        if (int rc = join()) return rc;
        const uint64_t n = of.size() - 1;
        if (n == 0) break;
        st->records += n;
        st->bases += used;
        adder = std::thread([&, n, b] {
            add_rc = ktb_counter_add(c, (const uint8_t *)hbases[b & 1].p, offs[b & 1].data(), n);
            if (add_rc) add_err = ktb_last_error();
        });
        if (parser.eof()) break;
    }
    return join();
}

// u32 counts of rows [r0, r1) -> "c0<d>c1<d>...\n" (format!("{}", f64) prints integral values without ".0", oligo.rs:138)
void format_counts_rows(const uint32_t *counts, uint64_t r0, uint64_t r1, uint32_t dim, char delim, Text *out) {
    out->resize((size_t)(r1 - r0) * dim * 11 + 16);
    char *o = out->data();
    size_t w = 0;
    for (uint64_t i = r0 * (uint64_t)dim; i < r1 * (uint64_t)dim; ++i) {
        uint32_t v = counts[i];
        char tmp[10];
        int len = 0;
        do { tmp[len++] = (char)('0' + v % 10); v /= 10; } while (v);
        while (len) o[w++] = tmp[--len];
        o[w++] = ((i + 1) % dim == 0) ? '\n' : delim;
    }
    out->resize(w);
}

// rows [0, n) cut into `threads` contiguous ranges, fn(r0, r1, part) run on one thread each (the `-t` of the CLI)
template <typename F>
void format_parallel(uint64_t n, int threads, std::vector<Text> *parts, F fn) {
    const uint64_t nt = std::max<uint64_t>(1, std::min<uint64_t>((uint64_t)threads, n));
    parts->resize(nt);
    if (nt == 1) { fn(0, n, &(*parts)[0]); return; }
    std::vector<std::thread> th;
    for (uint64_t t = 0; t < nt; ++t)
        th.emplace_back([&, t] { fn(n * t / nt, n * (t + 1) / nt, &(*parts)[t]); });
    for (auto &x : th) x.join();
}

// Rust's `{}` for f64: shortest digits that round-trip, never an exponent (std::to_chars fixed does the same).
// nullptr when the text does not fit in [o, end).
inline char *put_f64(char *o, char *end, double v) {
    auto r = std::to_chars(o, end, v, std::chars_format::fixed);
    return r.ec == std::errc() ? r.ptr : nullptr;
}

// Longest text of one CGR value.  A count is a u32: at most 10 digits.  A frequency c / t with 1 <= c <= t < 2^64 is
// 0, 1 or at least 2^-64 > 1e-20: "0." then at most 19 zeros before the first significant digit, and the shortest
// round-trip form of an f64 has at most 17 significant digits, so 38 characters.
constexpr size_t kCgrCountChars = 10;
constexpr size_t kCgrFreqChars = 2 + 19 + 17;

// composition/src/oligocgr.rs:123-143,165-190: every canonical k-mer gets a fixed point, the midpoint
// recurrence from the centre towards the corner of each base (A (0,0), T (v,0), G (v,v), C (0,v))
bool cgr_prefixes(const ktb_oligo *h, int k, uint64_t dim, double vecsize, std::vector<std::string> *pref) {
    std::vector<char> hb(dim * k);
    ktb_oligo_header(h, 1, hb.data(), hb.size());
    pref->resize(dim);
    for (uint64_t j = 0; j < dim; ++j) {
        double x = vecsize / 2.0, y = vecsize / 2.0;
        for (int i = 0; i < k; ++i) {
            double cx = 0, cy = 0;
            switch (hb[j * k + i]) {
                case 'A': cx = 0; cy = 0; break;
                case 'T': cx = vecsize; cy = 0; break;
                case 'G': cx = vecsize; cy = vecsize; break;
                default: cx = 0; cy = vecsize; break;  // 'C'
            }
            x = (cx + x) / 2.0;
            y = (cy + y) / 2.0;
        }
        char buf[900];
        char *o = buf;
        *o++ = '(';
        if (!(o = put_f64(o, buf + 440, x))) return false;
        *o++ = ',';
        if (!(o = put_f64(o, buf + 880, y))) return false;
        *o++ = ',';
        (*pref)[j].assign(buf, o);
    }
    return true;
}

// rows [r0, r1) -> "(x,y,freq) (x,y,freq) ...\n" (oligocgr.rs:88-101); false when a value's text exceeds its bound
bool format_cgr_rows(const void *rows, bool norm, uint64_t r0, uint64_t r1, uint32_t dim, const std::vector<std::string> &pref,
                     Text *out) {
    const size_t vmax = norm ? kCgrFreqChars : kCgrCountChars;
    size_t plen = 0;
    for (auto &p : pref) plen += p.size();
    out->resize((size_t)(r1 - r0) * (plen + (size_t)dim * (vmax + 2)));
    char *o = out->data();
    for (uint64_t i = r0; i < r1; ++i) {
        for (uint32_t j = 0; j < dim; ++j) {
            memcpy(o, pref[j].data(), pref[j].size());
            o += pref[j].size();
            if (norm) o = put_f64(o, o + vmax, ((const double *)rows)[i * dim + j]);
            else o = put_f64(o, o + vmax, (double)((const uint32_t *)rows)[i * dim + j]);
            if (!o) {
                out->clear();
                return false;
            }
            *o++ = ')';
            *o++ = (j + 1 == dim) ? '\n' : ' ';
        }
    }
    out->resize((size_t)(o - out->data()));
    return true;
}

// table entries [r0, r1) -> "<code>\t<count>\n", the code in decimal or (acgt) as k characters of ACGT
void format_count_lines(const uint64_t *keys, const uint64_t *counts, uint64_t r0, uint64_t r1, int k, bool acgt,
                        Text *out) {
    out->resize((size_t)(r1 - r0) * ((acgt ? (size_t)k : 20) + 22));
    char *o = out->data();
    for (uint64_t i = r0; i < r1; ++i) {
        if (acgt) {
            for (int j = 0; j < k; ++j) o[j] = "ACGT"[(keys[i] >> (2 * (k - 1 - j))) & 3u];
            o += k;
        } else {
            o = std::to_chars(o, o + 20, keys[i]).ptr;
        }
        *o++ = '\t';
        o = std::to_chars(o, o + 20, counts[i]).ptr;
        *o++ = '\n';
    }
    out->resize((size_t)(o - out->data()));
}

}  // namespace

extern "C" {

int ktb_debug_format6(double q, char *out8) {
    if (!out8 || !(q >= 0.0 && q <= 1.0)) return ktb_internal_fail(KTB_ERR_ARG, "format6 needs q in [0,1]");
    ktb::format6(q, out8);
    return KTB_OK;
}

void ktb_free(void *p) { free(p); }

int ktb_fastx_load(const char *path, int sniff, uint8_t **bases, uint64_t **offsets, uint64_t *n) {
    if (!path || !bases || !offsets || !n) return ktb_internal_fail(KTB_ERR_ARG, "null argument");
    *bases = nullptr; *offsets = nullptr; *n = 0;
    ktb::ByteSource src;
    std::string err;
    if (!src.open(path, &err)) return ktb_internal_fail(KTB_ERR_IO, err.c_str());
    ktb::SeqFormat fmt;
    if (sniff) {
        const int b = src.peek_first_byte();
        fmt = (b == '>') ? ktb::SeqFormat::Fasta : ktb::SeqFormat::Fastq;
        if (b < 0) { *offsets = (uint64_t *)calloc(1, 8); *bases = (uint8_t *)malloc(1); return KTB_OK; }
    } else if (!ktb::format_from_path(path, &fmt)) {
        return ktb_internal_fail(KTB_ERR_IO, "unknown sequence file extension (expected .fa/.fasta/.fna/.fq/.fastq[.gz])");
    }
    ktb::FastxParser parser(&src, fmt);
    std::vector<uint8_t> buf(1 << 20);
    std::vector<uint64_t> offs{0};
    size_t used = 0;
    for (;;) {
        const long r = parser.fill(buf.data(), buf.size(), &used, &offs, (size_t)1 << 40);
        if (r < 0) return ktb_internal_fail(KTB_ERR_IO, parser.error().c_str());
        if (parser.eof()) break;
        buf.resize(std::max(buf.size() * 2, used + parser.need_bytes() + 1024));
    }
    *n = offs.size() - 1;
    *bases = (uint8_t *)malloc(used ? used : 1);
    *offsets = (uint64_t *)malloc(offs.size() * 8);
    if (!*bases || !*offsets) return ktb_internal_fail(KTB_ERR_NOMEM, "malloc failed");
    if (used) memcpy(*bases, buf.data(), used);
    memcpy(*offsets, offs.data(), offs.size() * 8);
    return KTB_OK;
}

int ktb_debug_span_write(const char *path, const uint8_t *data, uint64_t len, uint64_t block, int threads, int mapped) {
    if (!path || (len && !data) || !block) return ktb_internal_fail(KTB_ERR_ARG, "bad argument");
    setenv("KTB_WRITER", mapped ? "map" : "seq", 1);
    ktb::SpanWriter wr;
    std::string err;
    const bool ok = wr.open(path, threads, &err);
    unsetenv("KTB_WRITER");
    if (!ok) return ktb_internal_fail(KTB_ERR_IO, err.c_str());
    std::vector<ktb::SpanWriter::Ticket> tickets((size_t)((len + block - 1) / block) + 1);
    size_t t = 0;
    for (uint64_t a = 0; a < len; a += block, ++t) wr.submit(data + a, (size_t)std::min(block, len - a), &tickets[t]);
    bool good = true;
    for (size_t i = 0; i < t; ++i) good &= wr.wait(&tickets[i]);
    if (wr.bytes() != len) good = false;
    if (!wr.close()) good = false;
    return good ? KTB_OK : ktb_internal_fail(KTB_ERR_IO, "write to the output file failed");
}

int ktb_debug_fastx_batches(const char *path, int sniff, uint64_t max_records, uint64_t batch_bytes, uint8_t **bases,
                            uint64_t **offsets, uint64_t *n) {
    if (!path || !bases || !offsets || !n || !max_records || !batch_bytes) return ktb_internal_fail(KTB_ERR_ARG, "bad argument");
    *bases = nullptr; *offsets = nullptr; *n = 0;
    ktb::ByteSource src;
    std::string err;
    if (!src.open(path, &err)) return ktb_internal_fail(KTB_ERR_IO, err.c_str());
    ktb::SeqFormat fmt;
    if (sniff) fmt = (src.peek_first_byte() == '>') ? ktb::SeqFormat::Fasta : ktb::SeqFormat::Fastq;
    else if (!ktb::format_from_path(path, &fmt)) return ktb_internal_fail(KTB_ERR_IO, "unknown sequence file extension");
    ktb::FastxParser parser(&src, fmt);
    std::vector<uint8_t> all, buf(batch_bytes);
    std::vector<uint64_t> all_offs{0}, offs;
    for (;;) {   // the batch loop of run_file, with caller-chosen batch limits
        offs.assign(1, 0);
        size_t used = 0;
        long got = 0;
        for (;;) {
            got = parser.fill(buf.data(), buf.size(), &used, &offs, (size_t)max_records);
            if (got < 0) return ktb_internal_fail(KTB_ERR_IO, parser.error().c_str());
            if (got == 0 && parser.need_bytes() && used == 0) {
                buf.resize(parser.need_bytes() + 16);
                continue;
            }
            break;
        }
        if (offs.size() == 1) break;
        for (size_t i = 1; i < offs.size(); ++i) all_offs.push_back(all.size() + offs[i]);
        all.insert(all.end(), buf.begin(), buf.begin() + used);
        if (parser.eof()) break;
    }
    *n = all_offs.size() - 1;
    *bases = (uint8_t *)malloc(all.size() ? all.size() : 1);
    *offsets = (uint64_t *)malloc(all_offs.size() * 8);
    if (!*bases || !*offsets) return ktb_internal_fail(KTB_ERR_NOMEM, "malloc failed");
    if (!all.empty()) memcpy(*bases, all.data(), all.size());
    memcpy(*offsets, all_offs.data(), all_offs.size() * 8);
    return KTB_OK;
}

// The counter and bins of `kmertools cov`, whose rows are coverage histograms of bin_count values.
struct CoverageRows {
    ktb_counter *c;
    uint32_t bin_size, bin_count;
};

// The drivers that write one line per record: `comp oligo` and `comp cgr` (k-mer rows of a ktb_oligo handle) and, with
// cov, `cov` (coverage rows of a counter).  Only the compute step of a batch differs between them.
static int run_file(const ktb_file_opts *o, ktb_file_stats *stats, int cgr_vecsize, const CoverageRows *cov = nullptr) {
    const bool cgr = cgr_vecsize > 0;
    const double t_start = now_ms();
    if (!o || !o->in_path || !o->out_path) return ktb_internal_fail(KTB_ERR_ARG, "null argument");
    ktb_file_stats st{};
    const bool norm = o->norm != 0;
    const std::string in = o->in_path;

    // ---- input + format (composition/src/oligo.rs:88-105,173)
    ktb::ByteSource src;
    std::string err;
    if (!src.open(in, &err)) return ktb_internal_fail(KTB_ERR_IO, err.c_str());
    ktb::SeqFormat fmt;
    if (in == "-" || !norm || cgr) {   // oligocgr.rs:64-72 always sniffs
        fmt = (src.peek_first_byte() == '>') ? ktb::SeqFormat::Fasta : ktb::SeqFormat::Fastq;
    } else if (!ktb::format_from_path(in, &fmt)) {
        return ktb_internal_fail(KTB_ERR_IO, "unknown sequence file extension (expected .fa/.fasta/.fna/.fq/.fastq[.gz])");
    }
    ktb::FastxParser parser(&src, fmt);

    ktb_oligo *h = nullptr;
    if (!cov)
        if (int rc = ktb_oligo_create(o->k, o->device, &h)) return rc;
    struct Guard { ktb_oligo *h; ~Guard() { ktb_oligo_destroy(h); } } guard{h};
    ktb::DeviceGuard device_guard(o->device);   // buffers and streams of this run live on the handle's device
    if (device_guard.err != cudaSuccess) return ktb_internal_fail(KTB_ERR_CUDA, "cudaSetDevice failed");
    const uint64_t dim = cov ? cov->bin_count : ktb_oligo_dim(h, cgr ? 1 : o->canonical);
    int sms = 0;
    if (h) sms = ktb_internal_sms(h);
    else if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, o->device) != cudaSuccess)
        return ktb_internal_fail(KTB_ERR_CUDA, "cudaDeviceGetAttribute failed");

    const int nthreads = host_threads(o->threads);
    ktb::SpanWriter wr;
    if (!wr.open(o->out_path, nthreads, &err)) return ktb_internal_fail(KTB_ERR_IO, err.c_str());
    ktb::SpanWriter::Ticket header_ticket;
    std::string header_line;

    std::vector<std::string> cgr_pref;
    if (cgr && !cgr_prefixes(h, o->k, dim, (double)cgr_vecsize, &cgr_pref))
        return ktb_internal_fail(KTB_ERR_ARG, "CGR coordinate text exceeds its bound");
    if (o->header && !cgr) {  // get_header().join(delim) + "\n", oligo.rs:114-117
        std::vector<char> hb(dim * o->k);
        if (int rc = ktb_oligo_header(h, o->canonical, hb.data(), hb.size())) return rc;
        std::string &line = header_line;
        line.reserve(dim * (o->k + 1));
        for (uint64_t j = 0; j < dim; ++j) {
            if (j) line.push_back(o->delim);
            line.append(hb.data() + j * o->k, o->k);
        }
        line.push_back('\n');
        wr.submit(line.data(), line.size(), &header_ticket);
    }

    // ---- batch geometry
    const bool gpu_text = norm && !cgr;          // fixed-width rows are formatted on the GPU
    const size_t out_per_row = gpu_text ? dim * 9 : ((cgr && norm) ? dim * 8 : dim * 4);
    // batches of 64 MB of output / 32 MB of bases: page-locking the two buffer sets is the fixed cost of a run
    // (~0.5 ms per MB; 1 GB of text: 752 ms -> 370 ms, 293 ms with the cached sets), and a batch this size already
    // hides every launch latency.
    // Round 1 measured 8 threads of pwrite per batch and dropped them (write()/pwrite() on one file serialise on the
    // inode lock); the writer now copies spans through a shared mapping instead, which does not.
    const size_t OUT_CAP = 64u << 20;
    const size_t max_records = std::max<size_t>(1, std::min<size_t>(OUT_CAP / out_per_row, 4u << 20));
    size_t bases_cap = input_bases_cap(in);

    SetPair *pair = acquire_sets(o->device);
    if (!pair) return ktb_internal_fail(KTB_ERR_CUDA, "cudaStreamCreate failed");
    struct PairGuard { SetPair *p; ~PairGuard() { release_sets(p); } } pair_guard{pair};
    // on every exit the writer threads stop BEFORE the buffer sets they read from go back to the pool
    struct WriterGuard { ktb::SpanWriter *w; ~WriterGuard() { w->close(); } } writer_guard{&wr};
    Set *sets = pair->sets;
    cudaEvent_t prev_kernels_done = nullptr;   // the handle's work counters / scratch are shared: kernels of
                                               // consecutive batches are chained, copies still overlap
    uint64_t launches = 0;
    double writer_wait_ms = 0;
    // the rows of a set are with the writer until its ticket completes; only then may its buffers be reused
    auto reclaim = [&](Set &s) -> int {
        if (!s.writing) return KTB_OK;
        const double t0 = now_ms();
        const bool ok = wr.wait(&s.ticket);
        writer_wait_ms += now_ms() - t0;
        s.writing = false;
        return ok ? KTB_OK : ktb_internal_fail(KTB_ERR_IO, "write to the output file failed");
    };

    auto finish = [&](Set &s) -> int {  // wait for the batch, write its rows
        if (!s.pending) return KTB_OK;
        const double t0 = now_ms();
        if (cudaStreamSynchronize(s.stream) != cudaSuccess)
            return ktb_internal_fail(KTB_ERR_CUDA, cudaGetErrorString(cudaGetLastError()));
        const double t1 = now_ms();
        st.gpu_wait_ms += t1 - t0;
        if (gpu_text) {
            wr.submit(s.h_out.p, s.out_bytes, &s.ticket);
        } else {
            const uint32_t *counts = (const uint32_t *)s.h_out.p;
            const void *rows = s.h_out.p;
            std::atomic<bool> text_ok{true};
            if (cgr)
                format_parallel(s.n, nthreads, &s.parts, [&](uint64_t r0, uint64_t r1, Text *part) {
                    if (!format_cgr_rows(rows, norm, r0, r1, (uint32_t)dim, cgr_pref, part)) text_ok = false;
                });
            else
                format_parallel(s.n, nthreads, &s.parts, [&](uint64_t r0, uint64_t r1, Text *part) {
                    format_counts_rows(counts, r0, r1, (uint32_t)dim, o->delim, part);
                });
            if (!text_ok) return ktb_internal_fail(KTB_ERR_IO, "CGR value text exceeds its bound");
            for (auto &part : s.parts) wr.submit(part.data(), part.size(), &s.ticket);
        }
        s.writing = true;
        st.write_ms += now_ms() - t1;
        s.pending = false;
        return KTB_OK;
    };

    // the compute step of one batch: u32 rows (f64 for normalised CGR rows) and totals of the batch on s.stream
    auto compute = [&](Set &s, bool f64rows) -> int {
        const uint8_t *d_bases = (const uint8_t *)s.d_bases.p;
        const uint64_t *d_offsets = (const uint64_t *)s.d_offsets.p;
        if (cov) {
            launches += 2;   // cov_hist_kernel, cov_write_kernel
            return ktb_counter_coverage_device(cov->c, d_bases, d_offsets, s.n, s.nbases, cov->bin_size, cov->bin_count,
                                               KTB_NORM_COUNTS, KTB_OUT_U32, s.d_counts.p, (uint64_t *)s.d_totals.p,
                                               s.stream);
        }
        const uint64_t l0 = ktb_internal_launches(h);
        const int rc = ktb_internal_dispatch(h, d_bases, d_offsets, s.n, s.nbases, cgr ? 1 : o->canonical,
                                             f64rows ? KTB_NORM_CLI : KTB_NORM_COUNTS, f64rows ? KTB_OUT_F64 : KTB_OUT_U32,
                                             s.d_counts.p, (uint64_t *)s.d_totals.p, s.stream);
        launches += ktb_internal_launches(h) - l0;
        return rc;
    };

    std::vector<uint64_t> offs;
    double alloc_ms = 0;   // page-locking / device allocation of the buffer sets (first two batches)
    const double t_loop = now_ms();
    int b = 0;
    for (;;) {
        Set &s = sets[b & 1];
        if (int rc = finish(s)) return rc;   // this set's previous batch (b-2) goes to the writer first ...
        if (int rc = reclaim(s)) return rc;  // ... and must have left the buffers
        const double ta0 = now_ms();
        if (!s.h_bases.ensure(bases_cap)) return ktb_internal_fail(KTB_ERR_NOMEM, "pinned allocation failed");
        const double tp0 = now_ms();
        alloc_ms += tp0 - ta0;
        size_t used = 0;
        if (int rc = fill_batch(parser, s.h_bases, &bases_cap, max_records, &used, &offs)) return rc;
        st.parse_ms += now_ms() - tp0;
        const uint64_t n = offs.size() - 1;
        if (n == 0) break;
        s.n = n;
        s.nbases = used;
        st.records += n;
        st.bases += used;
        // ---- enqueue H2D, kernels, D2H
        const double ta1 = now_ms();
        if (!s.h_offsets.ensure((n + 1) * 8)) return ktb_internal_fail(KTB_ERR_NOMEM, "pinned allocation failed");
        memcpy(s.h_offsets.p, offs.data(), (n + 1) * 8);
        s.out_bytes = n * out_per_row;
        if (!s.h_out.ensure(s.out_bytes) || !s.d_bases.ensure(used + 64) || !s.d_offsets.ensure((n + 1) * 8) ||
            !s.d_counts.ensure(n * dim * 8) || !s.d_totals.ensure(n * 8) || (gpu_text && !s.d_text.ensure(n * dim * 9)))
            return ktb_internal_fail(KTB_ERR_NOMEM, "buffer allocation failed");
        alloc_ms += now_ms() - ta1;
        cudaMemcpyAsync(s.d_bases.p, s.h_bases.p, used, cudaMemcpyHostToDevice, s.stream);
        cudaMemcpyAsync(s.d_offsets.p, s.h_offsets.p, (n + 1) * 8, cudaMemcpyHostToDevice, s.stream);
        if (prev_kernels_done) cudaStreamWaitEvent(s.stream, prev_kernels_done, 0);
        if (int rc = compute(s, cgr && norm)) return rc;   // CGR prints the f64 quotient itself ("{}")
        if (gpu_text) {
            const uint64_t nel = n * dim;
            uint64_t grid = (nel + 255) / 256;
            const uint64_t cap = (uint64_t)sms * 16;
            if (grid > cap) grid = cap;
            ktb::format_norm_kernel<<<(unsigned)grid, 256, 0, s.stream>>>(
                (const uint32_t *)s.d_counts.p, (const uint64_t *)s.d_totals.p, (uint8_t *)s.d_text.p, n, (uint32_t)dim,
                o->delim, KTB_NORM_CLI, o->canonical);
            ++launches;
            cudaEventRecord(s.kernels_done, s.stream);
            cudaMemcpyAsync(s.h_out.p, s.d_text.p, s.out_bytes, cudaMemcpyDeviceToHost, s.stream);
        } else {
            cudaEventRecord(s.kernels_done, s.stream);
            cudaMemcpyAsync(s.h_out.p, s.d_counts.p, s.out_bytes, cudaMemcpyDeviceToHost, s.stream);
        }
        prev_kernels_done = s.kernels_done;
        if (cudaGetLastError() != cudaSuccess) return ktb_internal_fail(KTB_ERR_CUDA, "enqueue failed");
        s.pending = true;
        ++b;
        if (parser.eof()) break;
    }
    // drain in order: the older batch first
    if (int rc = finish(sets[b & 1])) return rc;
    if (int rc = finish(sets[(b + 1) & 1])) return rc;
    if (int rc = reclaim(sets[b & 1])) return rc;
    if (int rc = reclaim(sets[(b + 1) & 1])) return rc;
    if (!wr.wait(&header_ticket)) return ktb_internal_fail(KTB_ERR_IO, "write to the output file failed");
    st.write_ms += writer_wait_ms;
    st.bytes_written = wr.bytes();
    const int wthreads = wr.threads();
    const bool wmapped = wr.mapped();
    if (!wr.close()) return ktb_internal_fail(KTB_ERR_IO, "closing the output file failed");
    st.launches = launches;
    st.total_ms = now_ms() - t_start;
    if (getenv("KTB_FILE_TRACE"))
        fprintf(stderr, "[ktb file] setup %.1f ms (handle, output file, streams), buffers %.1f ms, parse %.1f ms, gpu wait %.1f ms, "
                        "output %.1f ms on the caller (%.1f ms waiting for the %d %s writer thread(s)), total %.1f ms\n",
                t_loop - t_start, alloc_ms, st.parse_ms, st.gpu_wait_ms, st.write_ms, writer_wait_ms, wthreads,
                wmapped ? "mapping" : "sequential", st.total_ms);
    if (stats) *stats = st;
    return KTB_OK;
}

int ktb_comp_oligo_file(const ktb_file_opts *o, ktb_file_stats *stats) { return run_file(o, stats, 0); }

void ktb_release_cached_buffers(void) {
    SetPair *old = nullptr;
    {
        std::lock_guard<std::mutex> lk(g_pool_mutex);
        old = g_pool;
        g_pool = nullptr;
    }
    if (old) {
        ktb::DeviceGuard device_guard(old->device);
        delete old;
    }
}

int ktb_comp_cgr_file(const ktb_file_opts *o, int vecsize, ktb_file_stats *stats) {
    if (vecsize < 1) return ktb_internal_fail(KTB_ERR_ARG, "vecsize must be positive");
    return run_file(o, stats, vecsize);
}

int ktb_count_file(const ktb_file_opts *o, int acgt, ktb_file_stats *stats) {
    const double t_start = now_ms();
    if (!o || !o->in_path || !o->out_path) return ktb_internal_fail(KTB_ERR_ARG, "null argument");
    ktb_file_stats st{};
    const std::string in = o->in_path;
    ktb::ByteSource src;
    ktb::SeqFormat fmt;
    if (int rc = open_seq_input(in, &src, &fmt)) return rc;
    ktb::FastxParser parser(&src, fmt);

    ktb_counter *c = nullptr;
    if (int rc = ktb_counter_create(o->k, 1, o->device, &c)) return rc;
    struct Guard { ktb_counter *c; ~Guard() { ktb_counter_destroy(c); } } guard{c};
    ktb::DeviceGuard device_guard(o->device);   // page-locked buffers and the read-back stream belong to this device
    if (device_guard.err != cudaSuccess) return ktb_internal_fail(KTB_ERR_CUDA, "cudaSetDevice failed");
    std::error_code ec;
    std::filesystem::create_directories(o->out_path, ec);
    if (ec) return ktb_internal_fail(KTB_ERR_IO, ("cannot create the output directory: " + ec.message()).c_str());
    const std::string out_file = std::string(o->out_path) + "/kmers.counts";
    const int nthreads = host_threads(o->threads);

    if (int rc = count_into(c, parser, input_bases_cap(in), &st)) return rc;

    // ---- write: slices of the table through page-locked staging (slice s + 1 is copied while slice s is formatted)
    const double tw0 = now_ms();
    uint64_t nkeys = 0;
    ktb_counter_size(c, &nkeys, nullptr);
    const uint64_t *d_keys, *d_counts;
    ktb_internal_counter_table(c, &d_keys, &d_counts);
    std::string err;
    ktb::SpanWriter wr;
    if (!wr.open(out_file.c_str(), nthreads, &err)) return ktb_internal_fail(KTB_ERR_IO, err.c_str());
    const uint64_t SLICE = 1u << 22;
    struct Slice {
        Pinned keys, counts;
        std::vector<Text> parts;
        ktb::SpanWriter::Ticket ticket;
        bool writing = false;
    } sl[2];
    // on every exit the writer threads stop before the text they read goes away
    struct WriterGuard { ktb::SpanWriter *w; ~WriterGuard() { w->close(); } } writer_guard{&wr};
    cudaStream_t st_copy = nullptr;
    if (cudaStreamCreateWithFlags(&st_copy, cudaStreamNonBlocking) != cudaSuccess)
        return ktb_internal_fail(KTB_ERR_CUDA, "cudaStreamCreate failed");
    struct StreamGuard { cudaStream_t s; ~StreamGuard() { cudaStreamSynchronize(s); cudaStreamDestroy(s); } } stream_guard{st_copy};
    const uint64_t nslices = (nkeys + SLICE - 1) / SLICE;
    auto copy_out = [&](uint64_t si) -> int {
        Slice &x = sl[si & 1];
        const uint64_t a = si * SLICE, m = std::min(SLICE, nkeys - a);
        if (!x.keys.ensure(std::min(SLICE, nkeys) * 8) || !x.counts.ensure(std::min(SLICE, nkeys) * 8))
            return ktb_internal_fail(KTB_ERR_NOMEM, "pinned allocation failed");
        if (cudaMemcpyAsync(x.keys.p, d_keys + a, m * 8, cudaMemcpyDeviceToHost, st_copy) != cudaSuccess ||
            cudaMemcpyAsync(x.counts.p, d_counts + a, m * 8, cudaMemcpyDeviceToHost, st_copy) != cudaSuccess)
            return ktb_internal_fail(KTB_ERR_CUDA, "cudaMemcpyAsync(table slice) failed");
        return KTB_OK;
    };
    if (nslices)
        if (int rc = copy_out(0)) return rc;
    for (uint64_t si = 0; si < nslices; ++si) {
        Slice &x = sl[si & 1];
        if (cudaStreamSynchronize(st_copy) != cudaSuccess)
            return ktb_internal_fail(KTB_ERR_CUDA, cudaGetErrorString(cudaGetLastError()));
        if (si + 1 < nslices)   // the other slice's staging was formatted in the previous iteration
            if (int rc = copy_out(si + 1)) return rc;
        if (x.writing && !wr.wait(&x.ticket)) return ktb_internal_fail(KTB_ERR_IO, "write to the output file failed");
        const uint64_t m = std::min(SLICE, nkeys - si * SLICE);
        const uint64_t *keys = (const uint64_t *)x.keys.p, *counts = (const uint64_t *)x.counts.p;
        format_parallel(m, nthreads, &x.parts, [&](uint64_t r0, uint64_t r1, Text *part) {
            format_count_lines(keys, counts, r0, r1, o->k, acgt != 0, part);
        });
        for (auto &part : x.parts) wr.submit(part.data(), part.size(), &x.ticket);
        x.writing = true;
    }
    for (Slice &x : sl)
        if (x.writing && !wr.wait(&x.ticket)) return ktb_internal_fail(KTB_ERR_IO, "write to the output file failed");
    st.bytes_written = wr.bytes();
    if (!wr.close()) return ktb_internal_fail(KTB_ERR_IO, "closing the output file failed");
    st.write_ms = now_ms() - tw0;
    st.total_ms = now_ms() - t_start;
    if (stats) *stats = st;
    return KTB_OK;
}

int ktb_coverage_file(const ktb_file_opts *o, const char *count_path, uint32_t bin_size, uint32_t bin_count,
                      ktb_file_stats *stats) {
    const double t_start = now_ms();
    if (!o || !o->in_path || !o->out_path) return ktb_internal_fail(KTB_ERR_ARG, "null argument");
    if (o->k < 1 || o->k > KTB_MAX_SPARSE_K) {
        char msg[96];
        snprintf(msg, sizeof msg, "k must be in 1..%d for coverage rows (got %d)", KTB_MAX_SPARSE_K, o->k);
        return ktb_internal_fail(KTB_ERR_ARG, msg);
    }
    if (int rc = ktb_internal_coverage_args(bin_size, bin_count, KTB_NORM_COUNTS, KTB_OUT_U32)) return rc;
    const std::string in = o->in_path, counted = count_path ? count_path : o->in_path;
    if (in == "-" && counted == "-")
        return ktb_internal_fail(KTB_ERR_ARG, "stdin input needs a separate input to count (it would be read twice)");
    ktb::ByteSource src;
    ktb::SeqFormat fmt;
    if (int rc = open_seq_input(counted, &src, &fmt)) return rc;
    ktb::FastxParser parser(&src, fmt);

    ktb_counter *c = nullptr;
    if (int rc = ktb_counter_create(o->k, 1, o->device, &c)) return rc;
    struct Guard { ktb_counter *c; ~Guard() { ktb_counter_destroy(c); } } guard{c};
    ktb::DeviceGuard device_guard(o->device);   // page-locked buffers of the count pass belong to this device
    if (device_guard.err != cudaSuccess) return ktb_internal_fail(KTB_ERR_CUDA, "cudaSetDevice failed");
    ktb_file_stats count_st{};
    if (int rc = count_into(c, parser, input_bases_cap(counted), &count_st)) return rc;

    ktb_file_opts ro = *o;
    ro.canonical = 1;
    ro.norm = 1;
    ro.delim = ' ';
    ro.header = 0;
    const CoverageRows cov{c, bin_size, bin_count};
    ktb_file_stats st{};
    if (int rc = run_file(&ro, &st, 0, &cov)) return rc;
    st.parse_ms += count_st.parse_ms;
    st.gpu_wait_ms += count_st.gpu_wait_ms;
    st.total_ms = now_ms() - t_start;
    if (stats) *stats = st;
    return KTB_OK;
}

}  // extern "C"
