/*
 * kmertools_b200.h — C ABI of the B200-native oligonucleotide-frequency-vector path.
 *
 * This is the drop-in boundary for ONE hot path of anuradhawick/kmertools: per-sequence canonical
 * (or raw) k-mer counting + L1 normalisation.  The reference has no FFI seam of its own (it is a
 * single Rust process); the seam defined here is "batch of sequences -> dense row-major matrix",
 * which is exactly what its three callers consume:
 *
 *   composition/src/oligo.rs:231-259   OligoComputer::vectorise_one   (CLI, norm_mode 0/1)
 *   pybindings/src/oligo.rs:39-81      OligoComputer.vectorise_one / vectorise_batch (norm_mode 0/2)
 *   composition/src/oligocgr.rs:145-163 OligoCgrComputer::seq_to_kmer (same histogram)
 *
 * Plain pointers and sizes only.  All entry points return KTB_OK (0) or an error code; the message
 * is available from ktb_last_error() (thread-local).  Sequence CONTENT is never an error: ambiguous
 * bytes reset the k-mer window exactly as kmer/src/kmer.rs:80-106 does.
 *
 * There is NO CPU fallback: every compute entry point fails with KTB_ERR_NODEVICE when no CUDA device
 * is usable.
 */
#ifndef KMERTOOLS_B200_H
#define KMERTOOLS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KTB_ABI_VERSION 1

/* status codes */
#define KTB_OK 0
#define KTB_ERR_ARG 1      /* bad argument (k out of range, NULL pointer, unknown enum) */
#define KTB_ERR_CUDA 2     /* a CUDA call failed; see ktb_last_error() */
#define KTB_ERR_NOMEM 3    /* host or device allocation failed */
#define KTB_ERR_NODEVICE 4 /* no usable CUDA device */
#define KTB_ERR_IO 5       /* file could not be opened / parsed / written */

/* norm_mode: what vectorise_one does after counting.
 *   COUNTS  no normalisation                                  (oligo.rs:255 with norm=false)
 *   CLI     v[i] /= max(1, #kmers)                            (composition/src/oligo.rs:255-257)
 *   PY      like CLI, but in raw (non-canonical) mode the divisor is 2*#kmers, reproducing
 *           pybindings/src/oligo.rs:58-62 (`total += 2_f64`), so raw rows sum to 0.5 */
#define KTB_NORM_COUNTS 0
#define KTB_NORM_CLI 1
#define KTB_NORM_PY 2

/* out_dtype: element type of the output matrix.  U32 is only valid with KTB_NORM_COUNTS.
 * F64 reproduces the reference's Vec<f64> bit for bit; F32 is (float)(that f64 value). */
#define KTB_OUT_U32 0
#define KTB_OUT_F32 1
#define KTB_OUT_F64 2

/* largest k the dense-vector path supports (4^12/2 columns = 33.5 MB per f32 row) */
#define KTB_MAX_K 12

typedef struct ktb_oligo ktb_oligo;

/* Timings of the most recent vectorise call on a handle (milliseconds, CUDA events / host clock). */
typedef struct ktb_stats {
    double kernel_ms;      /* time during which a compute kernel of the call was running (chunks overlap: union, not sum) */
    double h2d_ms;         /* time during which a host->device copy was running (host-buffer entry point only) */
    double d2h_ms;         /* time during which a device->host copy was running */
    double wall_ms;        /* host wall clock of the whole call */
    uint64_t launches;     /* kernels launched by this library during the call */
    uint64_t h2d_bytes;
    uint64_t d2h_bytes;
} ktb_stats;

/* Number of CUDA devices visible to the library (0 when there is none / no driver). */
int ktb_device_count(void);

/* Replaces OligoComputer::new (composition/src/oligo.rs:31-47; pybindings/src/oligo.rs:22-31):
 * builds the canonical-rank tables of KmerGenerator::kmer_pos_maps (kmer/src/kmer.rs:54-73) and
 * uploads them to `device` (CUDA ordinal).  One handle per GPU; one process per GPU under torchrun.
 * 1 <= k <= KTB_MAX_K. */
int ktb_oligo_create(int k, int device, ktb_oligo **out);
void ktb_oligo_destroy(ktb_oligo *h);

int ktb_oligo_k(const ktb_oligo *h);
/* Row width: canonical -> |{min(x, rc(x))}| (kmer.rs:54-73), raw -> 4^k (oligo.rs:232-236). */
uint64_t ktb_oligo_dim(const ktb_oligo *h, int canonical);

/* Replaces OligoComputer::get_header (composition/src/oligo.rs:69-83; pybindings/src/oligo.rs:85-99):
 * dim labels of k characters each, written back to back (dim*k bytes, no separators, no NUL). */
int ktb_oligo_header(const ktb_oligo *h, int canonical, char *buf, size_t cap);

/* Replaces KmerGenerator::kmer_pos_maps (kmer/src/kmer.rs:54-73).  pos_map has 4^k entries
 * (canonical code -> rank, 0 elsewhere), pos_to_kmer has dim(canonical) entries.  Either may be NULL. */
int ktb_oligo_pos_maps(const ktb_oligo *h, uint64_t *pos_map, uint64_t *pos_to_kmer, uint64_t *count);

/* Replaces KmerGenerator::new + the whole iteration of KmerGenerator::next (kmer/src/kmer.rs:30-41,80-106;
 * pybindings/src/kmer.rs:22-44): every window of `seq` whose k bases are unambiguous, in position order, as the
 * forward code (first base most significant, A=0 C=1 G=2 T=3) and the code of its reverse complement.
 * 1 <= k <= 31 as in the reference.  HOST buffers; `*count` receives the number of valid windows, the first
 * min(*count, cap) pairs are written (cap = 0 with NULL arrays just counts; len - k + 1 always suffices). */
int ktb_kmer_pairs(const uint8_t *seq, uint64_t len, int k, int device, uint64_t *out_f, uint64_t *out_r,
                   uint64_t cap, uint64_t *count);

/* Same on DEVICE buffers of the current device, enqueued on `stream` (a cudaStream_t; NULL = default stream);
 * scratch comes from the stream-ordered allocator.  Returns after enqueueing.  *d_count is the full count (it may
 * exceed 2^32) whatever cap is; no element of d_out_f / d_out_r at or beyond min(*d_count, cap) is written.  d_seq
 * needs no alignment and may be NULL when len = 0; no byte outside [d_seq, d_seq + len) is read. */
int ktb_kmer_pairs_device(const uint8_t *d_seq, uint64_t len, int k, uint64_t *d_out_f, uint64_t *d_out_r,
                          uint64_t cap, uint64_t *d_count, void *stream);

/* Replaces OligoComputer::vectorise_one applied to a whole batch (pybindings vectorise_batch,
 * pybindings/src/oligo.rs:77-81; the rayon map in composition/src/oligo.rs:126-143).
 *
 * HOST-buffer entry point.  `bases` holds the sequences back to back (ASCII or raw 0..3 codes, as the
 * reference accepts), sequence i is bases[offsets[i] .. offsets[i+1]); offsets has n+1 entries.
 * `out` is n x dim row-major of out_dtype, caller-owned host memory (pinned memory from
 * ktb_host_alloc makes the copies asynchronous; pageable memory works too).  `totals` (optional, may
 * be NULL) receives the number of valid k-mer windows per sequence.  The call chunks the batch,
 * overlaps H2D / compute / D2H on CUDA streams and returns when `out` is complete. */
int ktb_oligo_vectorise(ktb_oligo *h, const uint8_t *bases, const uint64_t *offsets, uint64_t n,
                        int canonical, int norm_mode, int out_dtype, void *out, uint64_t *totals);

/* DEVICE-buffer entry point: same contract, but bases/offsets/out/totals are device pointers on the
 * handle's GPU and the work is enqueued on `stream` (a cudaStream_t; NULL = default stream).
 * Returns after enqueueing; results are ready when the stream reaches that point.
 * Offsets are absolute positions in d_bases: offsets[0] may be any value <= offsets[n], so a sub-batch view
 * (d_offsets + lo, n = hi - lo) of a batch resident in a larger buffer is valid input, at any offset.  total_bases must
 * equal offsets[n]: the call reads no byte of d_bases at or beyond it (a smaller value changes the rows).
 * d_bases and d_out must be 16-byte aligned.  The handle owns work counters and scratch buffers, so calls
 * on ONE handle must be ordered with respect to each other (same stream, or event-chained); use one handle
 * per concurrent stream.  Scratch buffers (reject lists, the pool of the bucket path, the order list of long contigs)
 * grow with cudaMalloc the first time a larger batch arrives, which synchronises the device once; steady-state calls of
 * the same or a smaller shape only enqueue. */
int ktb_oligo_vectorise_device(ktb_oligo *h, const uint8_t *d_bases, const uint64_t *d_offsets,
                               uint64_t n, uint64_t total_bases, int canonical, int norm_mode,
                               int out_dtype, void *d_out, uint64_t *d_totals, void *stream);

/* ---- sparse rows: per-sequence k-mer counts as CSR, 1 <= k <= KTB_MAX_SPARSE_K -------------------------------
 * The histogram of ktb_oligo_vectorise, stored as its non-zero entries.  For every sequence i and every valid window
 * (same decoding, validity and codes as ktb_kmer_pairs) key = min(forward, reverse complement) when canonical, the
 * forward code otherwise.  Row i holds every distinct key of sequence i in ascending order: codes[j] is the key (2-bit
 * code, A=0 C=1 G=2 T=3, first base most significant), values[j] its count as out_dtype with the normalisation of
 * the dense rows (the same divisor, the same f64 quotient, the same f32 rounding), so for k <= KTB_MAX_K scattering a
 * row through ktb_oligo_pos_maps (canonical) or by code (raw) gives the dense row bit for bit.  totals[i] = number of
 * valid windows.  Empty sequences, sequences shorter than k and all-ambiguous ones give empty rows.
 * Counts are 32-bit: a sequence must have fewer than 2^32 windows.  No handle: no tables are involved. */
#define KTB_MAX_SPARSE_K 31

/* HOST buffers.  row_ptr: n+1 entries, row_ptr[0] = 0, row i = entries [row_ptr[i], row_ptr[i+1]).
 * row_ptr (and totals, if not NULL) is always complete; codes / values are written only below cap
 * (cap = sum over sequences of max(0, len - k + 1) always suffices; cap = 0 with NULL arrays only sizes).
 * The batch is processed in chunks of whole sequences (about 2^26 bases each) on two streams: chunk c + 1 is copied
 * in and computed while the rows of chunk c are copied out (row_ptr and totals through page-locked staging).
 * A sequence with 2^32 or more windows is KTB_ERR_ARG. */
int ktb_sparse_vectorise(const uint8_t *bases, const uint64_t *offsets, uint64_t n, int k, int canonical,
                         int norm_mode, int out_dtype, int device, uint64_t *row_ptr, uint64_t *codes,
                         void *values, uint64_t cap, uint64_t *totals);

/* DEVICE buffers of the current device, enqueued on `stream` (a cudaStream_t; NULL = default stream); returns after
 * enqueueing, with no host round trip and no state shared between calls, so calls on different streams are
 * independent.  Offsets are absolute positions in d_bases as in ktb_oligo_vectorise_device (offsets[0] may be > 0);
 * total_bases must be at least offsets[n] (equal is the tightest): no byte at or beyond offsets[n] is read, and the
 * scratch is sized from total_bases.  d_row_ptr (n+1) and d_totals (n, may be NULL) are always complete; no element
 * of d_codes / d_values at or beyond cap is written.  Precondition: every sequence has fewer than 2^32 windows.
 * Scratch from the stream-ordered allocator: 24 bytes per base of total_bases (rounded up to 4096 bases) plus
 * 40 bytes per sequence.  The bases before offsets[0] count too: for a small batch deep inside a large buffer, pass
 * d_bases + offsets[0] with rebased offsets to keep the scratch small. */
int ktb_sparse_vectorise_device(const uint8_t *d_bases, const uint64_t *d_offsets, uint64_t n,
                                uint64_t total_bases, int k, int canonical, int norm_mode, int out_dtype,
                                uint64_t *d_row_ptr, uint64_t *d_codes, void *d_values, uint64_t cap,
                                uint64_t *d_totals, void *stream);

/* ---- batch-wide k-mer counting: one table of a whole data set, 1 <= k <= KTB_MAX_SPARSE_K ----------------------
 * Replaces CountComputer (`kmertools ctr`).  A counter has a fixed k and mode.  Adding a batch counts every valid
 * window of every sequence (same decoding, validity and codes as ktb_kmer_pairs), keyed by min(forward, reverse
 * complement) when canonical, by the forward code otherwise.  After any sequence of adds the table is every distinct
 * key seen, in ascending order, with a u64 count of its windows; it does not depend on how the input was split into
 * adds or on their order.  The sum of the counts is the number of valid windows added (nwindows).  Empty sequences,
 * sequences shorter than k and all-ambiguous ones contribute nothing.
 *
 * The table lives on the counter's device: 16 bytes per distinct key.  An add also needs scratch from the
 * stream-ordered allocator: 33 bytes per base of the batch (per base of total_bases for a device add; per base of a
 * chunk for a host add) plus, while the merge runs, the new table: 16 bytes per distinct key of the old table plus
 * 16 bytes per base (at most 16 * 4^k in all).  A host add of more than one chunk also holds the table it started
 * from, 16 bytes per key of it, until it returns.  A table or scratch that does not fit device memory is KTB_ERR_NOMEM
 * and leaves the counter as it was (a host add restores the table it started from, so none of the batch is counted);
 * nothing spills to the host or to disk.
 * Every add returns when the batch is in the table: it waits for its stream once, at the end, to learn the new table
 * size.  Calls on ONE counter must be ordered by the caller; different counters are independent. */
typedef struct ktb_counter ktb_counter;

/* 1 <= k <= KTB_MAX_SPARSE_K, canonical 0 or 1, device a CUDA ordinal.  Arguments are checked before any device work;
 * without a device the call is KTB_ERR_NODEVICE (there is no CPU path). */
int ktb_counter_create(int k, int canonical, int device, ktb_counter **out);
void ktb_counter_destroy(ktb_counter *c);

/* HOST buffers, layout of ktb_sparse_vectorise (offsets: n+1 entries, non-decreasing).  The batch is processed in
 * chunks of whole sequences (about 2^26 bases each; a longer sequence is a chunk of its own) on two streams of the
 * counter's device: chunk c + 1 is copied in while chunk c is counted and merged.  Returns when the batch is in the
 * table; synchronises only its own streams. */
int ktb_counter_add(ktb_counter *c, const uint8_t *bases, const uint64_t *offsets, uint64_t n);

/* DEVICE buffers on the counter's device, enqueued on `stream` (a cudaStream_t; NULL = default stream).  Offsets are
 * absolute positions in d_bases as in ktb_sparse_vectorise_device (offsets[0] may be > 0); total_bases must be at least
 * offsets[n]: no byte at or beyond offsets[n] is read, and the scratch is sized from total_bases (for a small batch
 * deep inside a large buffer, pass d_bases + offsets[0] with rebased offsets).  Waits for `stream` once, after the
 * merge, to read the new table size; the buffers may be reused when the call returns. */
int ktb_counter_add_device(ktb_counter *c, const uint8_t *d_bases, const uint64_t *d_offsets, uint64_t n,
                           uint64_t total_bases, void *stream);

/* Distinct keys of the table and valid windows added so far (either pointer may be NULL).  Every add has finished
 * when it returns, so this reads host fields and synchronises nothing. */
int ktb_counter_size(ktb_counter *c, uint64_t *nkeys, uint64_t *nwindows);

/* The first min(nkeys, cap) keys (ascending) and their counts into HOST memory; synchronous.  Nothing at or beyond
 * that index is written; cap = 0 writes nothing, and a NULL array is skipped. */
int ktb_counter_read(ktb_counter *c, uint64_t *keys, uint64_t *counts, uint64_t cap);

/* Same into DEVICE memory of the counter's device: device-to-device copies enqueued on `stream`, returns after
 * enqueueing.  The copies read the table in place, so the next add on the counter must be ordered after them: a
 * device add by its stream, a host add (which runs on streams of its own) by waiting for the copies on the host. */
int ktb_counter_read_device(ktb_counter *c, uint64_t *d_keys, uint64_t *d_counts, uint64_t cap, void *stream);

/* ---- per-read k-mer coverage histograms against a counter's table ---------------------------------------------
 * This build's own semantics (the reference's coverage tool is not reproduced).  For every sequence s of a batch and
 * every valid window of s (same decoding, validity and keys as the counter's adds: canonical or raw after the counter),
 * the window's abundance is a = the key's count in the table, or 0 when the key is absent (a table built from other
 * data).  Its bin is min(floor(a / bin_size), bin_count - 1), with a as u64.  Row s is the histogram of the bins of its
 * windows: bin_count u32 counts that sum to totals[s], the valid windows of s.  KTB_NORM_CLI divides each count by
 * max(1, totals[s]) exactly as the dense rows do (f64 the IEEE quotient, f32 that quotient rounded once);
 * KTB_NORM_COUNTS gives the counts (KTB_OUT_U32 needs it); KTB_NORM_PY is KTB_ERR_ARG.  Empty sequences, sequences
 * shorter than k and all-ambiguous ones give all-zero rows with total 0.  1 <= bin_size, 1 <= bin_count <= 65536; a
 * sequence must have fewer than 2^32 windows.  Arguments are checked before any device work.
 *
 * Lookups go through a directory over the top b bits of the 2k-bit key, b = floor(log2(distinct keys)) capped at 2k
 * (a direct index) and at 30: 8 * (2^b + 1) bytes on the counter's device, about half the table at most.  The first coverage call after an add
 * (or on a fresh counter) builds it and waits for its stream once; later calls only enqueue.  The next add frees it, as
 * does ktb_counter_destroy.  Each window then binary-searches one bucket of at most 2^(2k-b) keys.
 * Scratch: none per base; 4 bytes per row element with KTB_OUT_F64 (4-byte outputs are counted in place).  A directory
 * or scratch that does not fit device memory is KTB_ERR_NOMEM and leaves the counter usable. */

/* HOST buffers, layout of ktb_counter_add; chunks of whole sequences (about 2^26 bases each) on two streams, chunk c + 1
 * copied in and computed while the rows of chunk c are copied out.  out: n x bin_count row-major of out_dtype; totals
 * may be NULL (out too when n = 0).  Synchronous; a sequence with 2^32 or more windows is KTB_ERR_ARG. */
int ktb_counter_coverage(ktb_counter *c, const uint8_t *bases, const uint64_t *offsets, uint64_t n,
                         uint32_t bin_size, uint32_t bin_count, int norm_mode, int out_dtype,
                         void *out, uint64_t *totals);

/* DEVICE buffers on the counter's device, enqueued on `stream`; returns after enqueueing (after the directory build,
 * which waits for `stream`, on the first call after an add).  Offsets are absolute, total_bases >= offsets[n] as in
 * ktb_counter_add_device.  d_out (n x bin_count) and d_totals (n, may be NULL) are always complete.  The kernels read
 * the table and the directory in place, so the next add on the counter must be ordered after them: a device add by its
 * stream, a host add by waiting for them on the host (as for ktb_counter_read_device).  Once the directory exists a
 * coverage call changes nothing in the counter, so such calls may run concurrently on several streams.  Precondition:
 * every sequence has fewer than 2^32 windows. */
int ktb_counter_coverage_device(ktb_counter *c, const uint8_t *d_bases, const uint64_t *d_offsets, uint64_t n,
                                uint64_t total_bases, uint32_t bin_size, uint32_t bin_count, int norm_mode,
                                int out_dtype, void *d_out, uint64_t *d_totals, void *stream);

/* Stats of the most recent vectorise call (host entry point: complete; device entry point: launch
 * counts and class sizes only). */
int ktb_oligo_last_stats(const ktb_oligo *h, ktb_stats *out);

/* Tuning knobs (testing / benchmarking).  Known keys:
 *   "chunk_bytes"        target bytes of output per pipeline chunk in the host entry point
 *   "force_path"         0 auto, 1 flat-decomposition global-atomic kernel only, 2 no short-read kernel
 *   "seq_threads"        CTA size of the CTA-per-sequence kernel (0 = heuristic); each kernel clamps it to its own
 *                        launch bound: 1024 for the 32-bit rank-space histograms of k = 8, 256 everywhere else
 *   "seq_grab"           sequences a CTA of that kernel takes per trip to the work counter (0 = heuristic)
 *   "dense_odd"          1 (default): dense middle-base histogram for k = 7 in seq_kernel (mode 4), 0: code-space histogram
 *   "even_rank"          1 (default): even k whose rank-space histogram fits shared memory (k = 8) compute the rank from two
 *                        small shared-memory tables (seq_kernel mode 7 / 5, long_kernel MODE_K8); 0: rank table in L2 (mode 2)
 *   "packed16"           1 (default): 16-bit counters packed two to a word for k = 8 (three CTAs per SM; sequences with more
 *                        than 65535 windows take a second launch with 32-bit counters); 0: 32-bit rank-space histogram
 *   "k8_long"            1 (default): k = 8 u32 / f32 rows are counted by long_kernel MODE_K8; 0: seq_kernel mode 5
 *   "k7_mid"             1 (default): k = 7 rows by long_kernel (middle-base-first keys, scheduled write-out); 0: seq_kernel
 *   "fwd_fold"           1 (default): 3 <= k <= 5 rows of long sequences by long_kernel (forward codes folded at write-out)
 *   "fwd_min_len"        mean sequence length from which "fwd_fold" applies (default 1024)
 *   "fwd_replicas"       1 (default): long contigs (mean length >= 32 kbp) at k <= 5 count into lane-private replicas of the bins
 *   "longest_first"      1 (default): such batches of long contigs are handed to the CTAs longest length class first;
 *                        0: input order
 *   "long_warps"         warps per CTA of long_kernel (0 = heuristic; 4, 8 or 10)
 *   "bucket"             1 (default): rows larger than shared memory (canonical k = 9, 10; raw k = 8..10) are built by
 *                        bucket_kernel + count_kernel (partition by code segment, count in shared memory); 0: wave_kernel
 *   "bucket_log2_seg"    log2 of the codes per segment of that path (13 or 14, default 14)
 *   "bucket_hist_kb"     histogram memory of count_kernel per CTA: 64 (default, three CTAs per SM) or 96 (two CTAs, more
 *                        segments alternate between two buffers)
 *   "bucket_waves"       waves of that path (bucket_kernel of wave w+1 beside count_kernel of wave w; default 1 = off,
 *                        measured best) and "bucket_wave_ctas" (bucket_kernel CTAs per SM in wave mode, 1..4, default 2)
 *   "wave_persistent"    1 (default): where the bucket path does not apply (k >= 11, or "bucket" = 0) histograms larger than
 *                        shared memory are counted by one cooperative launch for u32 / f32 output; 0: one memset + kernel
 *                        (+ normalise) per wave
 *   "wave_smem_rank"     1 (default): that kernel computes canonical ranks from shared-memory tables (k <= 10)
 *   "wave_budget_bytes"  L2 budget of that kernel; a wave (rows zeroed, counted and normalised together) is a third of it
 *   "global_wave_bytes"  bytes of output rows zeroed + counted together by the multi-launch variant (fits L2)
 *   "global_steps_per_warp"  granularity of that variant's work items: steps of 512 bases per warp (default 1) */
int ktb_oligo_set_option(ktb_oligo *h, const char *key, int64_t value);

/* Pinned host memory for callers that want asynchronous copies (usable from every device).  ktb_host_alloc_near binds
 * the pages to the NUMA node of `device` (from /sys/bus/pci/devices/<bdf>/numa_node; falls back to ktb_host_alloc when
 * the topology is unknown), so that the copies of several GPUs do not all land on one node.  ktb_host_free frees both. */
void *ktb_host_alloc(size_t bytes);
void *ktb_host_alloc_near(size_t bytes, int device);
void ktb_host_free(void *p);
/* NUMA node of a CUDA device, -1 when unknown. */
int ktb_device_numa_node(int device);

/* ---- several GPUs, one call (SURVEY.md §8e) --------------------------------------------------------------------
 * Replaces the reference's fan-out of ONE batch over all its workers with the row order kept
 * (composition/src/oligo.rs:126-143 `buffer.par_iter().map(..).collect()`, pybindings/src/oligo.rs:77-81
 * `seqs.into_par_iter()`): the batch is cut into one contiguous range of sequences per device, balanced by bases;
 * every device computes its rows from its own host thread (one ktb_oligo handle, three stream sets per device) and
 * writes its own slab of `out`.  Rows are independent: no collective.  ndev = 0 takes every visible device. */
typedef struct ktb_multi ktb_multi;
int ktb_multi_create(int k, const int *devices, int ndev, ktb_multi **out);
void ktb_multi_destroy(ktb_multi *m);
int ktb_multi_device_count(const ktb_multi *m);
/* The per-device handle (for ktb_oligo_set_option / ktb_oligo_dim / ktb_oligo_header); owned by `m`. */
ktb_oligo *ktb_multi_handle(ktb_multi *m, int i);
/* Same contract as ktb_oligo_vectorise (host buffers). */
int ktb_multi_vectorise(ktb_multi *m, const uint8_t *bases, const uint64_t *offsets, uint64_t n, int canonical,
                        int norm_mode, int out_dtype, void *out, uint64_t *totals);
/* Stats and row range [first_row, end_row) of device i in the most recent ktb_multi_vectorise. */
int ktb_multi_last_stats(const ktb_multi *m, int i, ktb_stats *out, uint64_t *first_row, uint64_t *end_row);
/* Page-locked n x dim output whose slab of device i lives on that device's NUMA node (release with ktb_host_free). */
void *ktb_multi_alloc_rows(const ktb_multi *m, const uint64_t *offsets, uint64_t n, int canonical, int out_dtype);
/* The partition itself: bounds[0..parts], part r = sequences [bounds[r], bounds[r+1]); cut r is the first sequence that
 * starts at or after r/parts of the bases (by count when every sequence is empty).  Pure host arithmetic. */
int ktb_shard_bounds(const uint64_t *offsets, uint64_t n, int parts, uint64_t *bounds);

/* ---- file-level driver: `kmertools comp oligo` (kmertools/src/args.rs:70-103,242-263) ---------------
 * Replaces OligoComputer::{new, set_*, vectorise} (composition/src/oligo.rs:31-229): reads FASTA/FASTQ
 * (optionally .gz, "-" = stdin; ktio/src/seq.rs:29-155), computes the rows on the GPU and writes the
 * same text the reference writes: header row (optional), one line per record, values "{:.6}" when
 * normalising (formatted on the GPU) or integer counts, joined by `delim`.
 * Format detection follows oligo.rs:88-105,173: stdin or counts mode sniff the first byte, otherwise
 * the extension decides (unknown extension is an error; the reference panics there). */
typedef struct ktb_file_opts {
    const char *in_path;   /* "-" = stdin */
    const char *out_path;
    int k;                 /* args.rs restricts the CLI to 3..=7; the library accepts 1..KTB_MAX_K */
    int canonical;         /* count_min = !raw_count */
    int norm;              /* !counts */
    char delim;            /* ' ', ',' or '\t' */
    int header;
    int threads;           /* accepted for CLI compatibility; host formatting threads for counts mode */
    int device;            /* CUDA ordinal */
} ktb_file_opts;

typedef struct ktb_file_stats {
    uint64_t records;
    uint64_t bases;
    uint64_t bytes_written;
    double parse_ms, gpu_wait_ms, write_ms, total_ms;
    uint64_t launches;
} ktb_file_stats;

int ktb_comp_oligo_file(const ktb_file_opts *opts, ktb_file_stats *stats /* optional */);

/* `kmertools comp cgr -k K` (k-mer mode; OligoCgrComputer, composition/src/oligocgr.rs:63-163): the same
 * canonical histogram, printed as "(x,y,freq)" triples where (x,y) is the fixed chaos-game point of the
 * column's k-mer in a vecsize x vecsize square.  Uses in_path, out_path, k, norm, device of `opts`. */
int ktb_comp_cgr_file(const ktb_file_opts *opts, int vecsize, ktb_file_stats *stats /* optional */);

/* `kmertools ctr`: the canonical k-mer counts of a whole file (ktb_counter_*, 1 <= k <= KTB_MAX_SPARSE_K).  Uses
 * in_path, out_path, k, threads and device of `opts`; the input format follows ktb_comp_oligo_file (the extension
 * decides, "-" = stdin sniffs the first byte).  The file is parsed in batches into one counter, parsing batch b + 1
 * while batch b is added.  out_path is a directory, created if missing; the table is written to out_path/kmers.counts,
 * one line per distinct k-mer in ascending code order: "<code>\t<count>\n" with the code in decimal, or with acgt != 0
 * the k-mer as k characters of ACGT (first base first).  The table is read back in slices through page-locked staging
 * and formatted by `threads` host threads.  stats->bases counts the bases parsed, stats->bytes_written the text. */
int ktb_count_file(const ktb_file_opts *opts, int acgt, ktb_file_stats *stats /* optional */);

/* `kmertools cov`: counts the canonical k-mers of count_path (NULL = in_path) into a counter, then writes one line per
 * record of in_path: the record's coverage histogram (ktb_counter_coverage, KTB_NORM_CLI), bin_count values "{:.6}"
 * joined by ' ', '\n'-terminated, in input order.  Uses in_path, out_path, k, threads, device of opts.  Both inputs
 * follow ktb_count_file's format rule; in_path "-" (stdin) needs a count_path other than "-", since the input would be
 * read twice.  k, bin_size, bin_count and that rule are checked before any device work.  The line form is this build's
 * own.  stats describe the second pass (records and bases of in_path). */
int ktb_coverage_file(const ktb_file_opts *opts, const char *count_path, uint32_t bin_size, uint32_t bin_count,
                      ktb_file_stats *stats /* optional */);

/* The file-level drivers keep their pinned / device buffer sets (at most ~0.5 GB) for the next call on the same
 * device; this frees them. */
void ktb_release_cached_buffers(void);

/* Loads a whole FASTA/FASTQ(.gz) file into packed buffers (malloc'ed; release with ktb_free).
 * sniff != 0: format from the first byte, else from the extension. */
int ktb_fastx_load(const char *path, int sniff, uint8_t **bases, uint64_t **offsets, uint64_t *n);
void ktb_free(void *p);

/* ktb_fastx_load through the BATCH loop of the file-level drivers (at most max_records records and batch_bytes bytes of
 * sequence per batch), so tests can put batch boundaries anywhere in a file.  Same outputs as ktb_fastx_load. */
int ktb_debug_fastx_batches(const char *path, int sniff, uint64_t max_records, uint64_t batch_bytes, uint8_t **bases,
                            uint64_t **offsets, uint64_t *n);

/* The output writer of the file-level drivers on its own (csrc/span_writer.h): `data` goes to `path` in blocks of `block`
 * bytes, asynchronously, by `threads` threads through a shared mapping (mapped != 0) or by one thread with write(). */
int ktb_debug_span_write(const char *path, const uint8_t *data, uint64_t len, uint64_t block, int threads, int mapped);

/* Host build of the GPU text formatter: 8 characters "d.dddddd" = Rust's format!("{:.6}", q), q in [0,1]. */
int ktb_debug_format6(double q, char *out8);

/* Device byte -> 2-bit code table as the kernels compute it (256 entries); lets tests compare the
 * in-kernel decoder with SEQ_NT4_TABLE (kmer/src/kmer.rs:6-15). */
int ktb_debug_nt4_table(ktb_oligo *h, uint8_t *out256);

const char *ktb_last_error(void);
int ktb_abi_version(void);

#ifdef __cplusplus
}
#endif
#endif /* KMERTOOLS_B200_H */
