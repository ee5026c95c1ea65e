// kmertools — drop-in for the reference CLI's `comp oligo` subcommand (kmertools/src/args.rs:70-103,
// 242-263).  Same flags, same defaults, same output bytes; compute runs on the GPU through
// libkmertools_b200.so.  Also `comp cgr -k`, `ctr` (batch-wide k-mer counts, with this build's own output file) and
// `cov` (per-record k-mer coverage histograms, this build's own semantics and output).
// Other subcommands of the reference are out of scope (SURVEY.md §2).
#include "../../../include/kmertools_b200.h"

#include <cerrno>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>

static void usage() {
    fprintf(stderr,
            "Generate oligonucleotide frequency vectors (GPU)\n\n"
            "Usage: kmertools comp oligo [OPTIONS] --input <INPUT> --output <OUTPUT>\n\n"
            "Options:\n"
            "  -i, --input <INPUT>    Input file path\n"
            "  -o, --output <OUTPUT>  Output vectors path\n"
            "  -c, --counts           Disable normalisation and output raw counts\n"
            "  -k, --k-size <K_SIZE>  Set k-mer size [default: 3]\n"
            "  -r, --raw-count        Raw counts\n"
            "  -p, --preset <PRESET>  Output type to write [default: spc] [possible values: csv, tsv, spc]\n"
            "  -H, --header           Include header (with k-mer in ACGT format)\n"
            "  -t, --threads <N>      Thread count for computations 0=auto [default: 0]\n"
            "      --device <N>       CUDA device ordinal [default: 0]\n");
}

// `kmertools comp cgr -k K ...` (k-mer mode of kmertools/src/args.rs:105-128,264-283)
static int main_cgr(int argc, char **argv) {
    ktb_file_opts o{};
    std::string in, out;
    o.k = 0; o.canonical = 1; o.norm = 1; o.delim = ' '; o.device = 0;
    long vec = -1;
    for (int i = 3; i < argc; ++i) {
        const std::string a = argv[i];
        auto val = [&](const char *name) -> const char * {
            if (i + 1 >= argc) { fprintf(stderr, "error: a value is required for '%s'\n", name); exit(2); }
            return argv[++i];
        };
        if (a == "-i" || a == "--input") in = val("--input");
        else if (a == "-o" || a == "--output") out = val("--output");
        else if (a == "-c" || a == "--counts") o.norm = 0;
        else if (a == "-k" || a == "--k-size") o.k = atoi(val("--k-size"));
        else if (a == "-v" || a == "--vec-size") vec = atol(val("--vec-size"));
        else if (a == "-t" || a == "--threads") o.threads = atoi(val("--threads"));
        else if (a == "--device") o.device = atoi(val("--device"));
        else { fprintf(stderr, "error: unexpected argument '%s' found\n", a.c_str()); return 2; }
    }
    if (in.empty() || out.empty()) { fprintf(stderr, "error: --input and --output are required\n"); return 2; }
    if (o.k == 0) {
        fprintf(stderr, "error: whole-sequence CGR (no -k) is outside this build's scope; use -k 3..7 for k-mer mode\n");
        return 2;
    }
    if (o.k < 3 || o.k > 7) {
        fprintf(stderr, "error: invalid value '%d' for '--k-size <K_SIZE>': %d is not in 3..=7\n", o.k, o.k);
        return 2;
    }
    if (vec < 0) vec = (long)(o.k * o.k);   // (k as f64).powf(4.0).powf(0.5) as u64
    o.in_path = in.c_str();
    o.out_path = out.c_str();
    if (ktb_comp_cgr_file(&o, (int)vec, nullptr) != KTB_OK) fprintf(stderr, "Error: %s\n", ktb_last_error());
    return 0;
}

static void usage_ctr() {
    fprintf(stderr,
            "Count the canonical k-mers of a whole file (GPU)\n\n"
            "Usage: kmertools ctr [OPTIONS] --input <INPUT> --output <OUTPUT> --k-size <K_SIZE>\n\n"
            "Writes OUTPUT/kmers.counts (OUTPUT is a directory, created if missing): one line per distinct canonical\n"
            "k-mer, min(forward, reverse complement), in ascending code order, as \"<code>\\t<count>\\n\" with the 2-bit\n"
            "code (A=0 C=1 G=2 T=3, first base most significant) in decimal.  The file name and line form are this\n"
            "build's own; the reference writes its counts in another order.\n\n"
            "Options:\n"
            "  -i, --input <INPUT>    Input file path (FASTA/FASTQ by extension, optionally .gz; - = stdin)\n"
            "  -o, --output <OUTPUT>  Output directory\n"
            "  -k, --k-size <K_SIZE>  k-mer size, 10..=31\n"
            "  -m, --memory <GB>      Accepted and ignored: the table lives in GPU memory\n"
            "  -a, --acgt             Write each k-mer as k characters of ACGT instead of its code\n"
            "  -t, --threads <N>      Threads formatting and writing the output 0=auto [default: 0]\n"
            "      --device <N>       CUDA device ordinal [default: 0]\n"
            "      --any-k            Accept any k in 1..=31\n"
            "  -h, --help             Print help\n");
}

// `kmertools ctr`: batch-wide canonical k-mer counts (CountComputer)
static int main_ctr(int argc, char **argv) {
    ktb_file_opts o{};
    std::string in, out;
    o.k = 0; o.canonical = 1; o.delim = '\t'; o.device = 0;
    int acgt = 0;
    bool any_k = false, have_k = false;
    for (int i = 2; i < argc; ++i) {
        const std::string a = argv[i];
        auto val = [&](const char *name) -> const char * {
            if (i + 1 >= argc) { fprintf(stderr, "error: a value is required for '%s'\n", name); exit(2); }
            return argv[++i];
        };
        if (a == "-i" || a == "--input") in = val("--input");
        else if (a == "-o" || a == "--output") out = val("--output");
        else if (a == "-k" || a == "--k-size") { o.k = atoi(val("--k-size")); have_k = true; }
        else if (a == "-m" || a == "--memory") val("--memory");
        else if (a == "-a" || a == "--acgt") acgt = 1;
        else if (a == "-t" || a == "--threads") o.threads = atoi(val("--threads"));
        else if (a == "--device") o.device = atoi(val("--device"));
        else if (a == "--any-k") any_k = true;
        else if (a == "-h" || a == "--help") { usage_ctr(); return 0; }
        else { fprintf(stderr, "error: unexpected argument '%s' found\n", a.c_str()); usage_ctr(); return 2; }
    }
    if (in.empty() || out.empty() || !have_k) {
        fprintf(stderr, "error: the following required arguments were not provided:\n%s%s%s", in.empty() ? "  --input <INPUT>\n" : "",
                out.empty() ? "  --output <OUTPUT>\n" : "", have_k ? "" : "  --k-size <K_SIZE>\n");
        return 2;
    }
    const int lo = any_k ? 1 : 10;
    if (o.k < lo || o.k > 31) {
        fprintf(stderr, "error: invalid value '%d' for '--k-size <K_SIZE>': %d is not in %d..=31\n", o.k, o.k, lo);
        return 2;
    }
    o.in_path = in.c_str();
    o.out_path = out.c_str();
    ktb_file_stats st{};
    if (ktb_count_file(&o, acgt, &st) != KTB_OK) {
        fprintf(stderr, "Error: %s\n", ktb_last_error());   // exit 0, as for `comp oligo` (args.rs:260-262)
        return 0;
    }
    if (getenv("KTB_VERBOSE"))
        fprintf(stderr, "records %llu bases %llu written %llu B | parse %.1f ms add-wait %.1f ms write %.1f ms total %.1f ms\n",
                (unsigned long long)st.records, (unsigned long long)st.bases, (unsigned long long)st.bytes_written,
                st.parse_ms, st.gpu_wait_ms, st.write_ms, st.total_ms);
    return 0;
}

static void usage_cov() {
    fprintf(stderr,
            "Per-record k-mer coverage histograms (GPU)\n\n"
            "Usage: kmertools cov [OPTIONS] --input <INPUT> --output <OUTPUT>\n\n"
            "Counts the canonical k-mers of COUNT_IN (default: INPUT) on the GPU, then writes one line per record of INPUT:\n"
            "BIN_COUNT values \"{:.6}\" joined by ' '.  Value b is the share of the record's valid k-mer windows whose\n"
            "k-mer has a count a in the table with min(floor(a / BIN_SIZE), BIN_COUNT - 1) = b (a = 0 for k-mers absent\n"
            "from it).  The semantics and the line form are this build's own.\n\n"
            "Options:\n"
            "  -i, --input <INPUT>        Input file path (FASTA/FASTQ by extension, optionally .gz; - = stdin, needs -a)\n"
            "  -o, --output <OUTPUT>      Output file path\n"
            "  -a, --abundance <COUNT_IN> Sequences whose k-mers are counted (same formats; - = stdin) [default: INPUT]\n"
            "  -k, --k-size <K_SIZE>      k-mer size, 10..=31 [default: 15]\n"
            "  -w, --bin-size <BIN_SIZE>  Counts per bin, at least 1 [default: 16]\n"
            "  -c, --bin-count <COUNT>    Bins per line, 1..=65536; the last one takes every larger count [default: 16]\n"
            "  -m, --memory <GB>          Accepted and ignored: the table lives in GPU memory\n"
            "  -t, --threads <N>          Threads writing the output 0=auto [default: 0]\n"
            "      --device <N>           CUDA device ordinal [default: 0]\n"
            "      --any-k                Accept any k in 1..=31\n"
            "  -h, --help                 Print help\n");
}

// a whole decimal number in [lo, hi], or -1
static long long parse_count(const char *s, long long lo, long long hi) {
    char *end = nullptr;
    errno = 0;
    const long long v = strtoll(s, &end, 10);
    if (errno || end == s || *end || v < lo || v > hi) return -1;
    return v;
}

// `kmertools cov`: per-record coverage histograms against the k-mer counts of a whole file
static int main_cov(int argc, char **argv) {
    ktb_file_opts o{};
    std::string in, out, counted;
    bool have_counted = false, any_k = false;
    o.k = 15; o.canonical = 1; o.norm = 1; o.delim = ' '; o.device = 0;
    long long bin_size = 16, bin_count = 16;
    for (int i = 2; i < argc; ++i) {
        const std::string a = argv[i];
        auto val = [&](const char *name) -> const char * {
            if (i + 1 >= argc) { fprintf(stderr, "error: a value is required for '%s'\n", name); exit(2); }
            return argv[++i];
        };
        if (a == "-i" || a == "--input") in = val("--input");
        else if (a == "-o" || a == "--output") out = val("--output");
        else if (a == "-a" || a == "--abundance") { counted = val("--abundance"); have_counted = true; }
        else if (a == "-k" || a == "--k-size") o.k = atoi(val("--k-size"));
        else if (a == "-w" || a == "--bin-size") {
            const char *v = val("--bin-size");
            if ((bin_size = parse_count(v, 1, 0xFFFFFFFFll)) < 0) {
                fprintf(stderr, "error: invalid value '%s' for '--bin-size <BIN_SIZE>': not in 1..=4294967295\n", v);
                return 2;
            }
        } else if (a == "-c" || a == "--bin-count") {
            const char *v = val("--bin-count");
            if ((bin_count = parse_count(v, 1, 65536)) < 0) {
                fprintf(stderr, "error: invalid value '%s' for '--bin-count <COUNT>': not in 1..=65536\n", v);
                return 2;
            }
        }
        else if (a == "-m" || a == "--memory") val("--memory");
        else if (a == "-t" || a == "--threads") o.threads = atoi(val("--threads"));
        else if (a == "--device") o.device = atoi(val("--device"));
        else if (a == "--any-k") any_k = true;
        else if (a == "-h" || a == "--help") { usage_cov(); return 0; }
        else { fprintf(stderr, "error: unexpected argument '%s' found\n", a.c_str()); usage_cov(); return 2; }
    }
    if (in.empty() || out.empty()) {
        fprintf(stderr, "error: the following required arguments were not provided:\n%s%s", in.empty() ? "  --input <INPUT>\n" : "",
                out.empty() ? "  --output <OUTPUT>\n" : "");
        return 2;
    }
    const int lo = any_k ? 1 : 10;
    if (o.k < lo || o.k > 31) {
        fprintf(stderr, "error: invalid value '%d' for '--k-size <K_SIZE>': %d is not in %d..=31\n", o.k, o.k, lo);
        return 2;
    }
    if (in == "-" && (!have_counted || counted == "-")) {
        fprintf(stderr, "error: --input - (stdin) needs --abundance <COUNT_IN> from another source: the input would be read twice\n");
        return 2;
    }
    o.in_path = in.c_str();
    o.out_path = out.c_str();
    ktb_file_stats st{};
    if (ktb_coverage_file(&o, have_counted ? counted.c_str() : nullptr, (uint32_t)bin_size, (uint32_t)bin_count, &st) != KTB_OK) {
        fprintf(stderr, "Error: %s\n", ktb_last_error());   // exit 0, as for `comp oligo` (args.rs:260-262)
        return 0;
    }
    if (getenv("KTB_VERBOSE"))
        fprintf(stderr, "records %llu bases %llu written %llu B | parse %.1f ms gpu-wait %.1f ms write %.1f ms total %.1f ms\n",
                (unsigned long long)st.records, (unsigned long long)st.bases, (unsigned long long)st.bytes_written,
                st.parse_ms, st.gpu_wait_ms, st.write_ms, st.total_ms);
    return 0;
}

int main(int argc, char **argv) {
    if (argc >= 2 && !strcmp(argv[1], "ctr")) return main_ctr(argc, argv);
    if (argc >= 2 && !strcmp(argv[1], "cov")) return main_cov(argc, argv);
    if (argc >= 3 && !strcmp(argv[1], "comp") && !strcmp(argv[2], "cgr")) return main_cgr(argc, argv);
    if (argc < 3 || strcmp(argv[1], "comp") != 0 || strcmp(argv[2], "oligo") != 0) {
        if (argc >= 2 && (!strcmp(argv[1], "-h") || !strcmp(argv[1], "--help"))) { usage(); return 0; }
        fprintf(stderr, "error: this build provides only `kmertools comp oligo`, `kmertools comp cgr -k`, `kmertools ctr` and `kmertools cov`\n");
        usage();
        return 2;
    }
    ktb_file_opts o{};
    std::string in, out;
    o.k = 3; o.canonical = 1; o.norm = 1; o.delim = ' '; o.header = 0; o.threads = 0; o.device = 0;
    bool k_range_checked = true;
    for (int i = 3; i < argc; ++i) {
        const std::string a = argv[i];
        auto val = [&](const char *name) -> const char * {
            if (i + 1 >= argc) { fprintf(stderr, "error: a value is required for '%s'\n", name); exit(2); }
            return argv[++i];
        };
        if (a == "-i" || a == "--input") in = val("--input");
        else if (a == "-o" || a == "--output") out = val("--output");
        else if (a == "-c" || a == "--counts") o.norm = 0;
        else if (a == "-k" || a == "--k-size") o.k = atoi(val("--k-size"));
        else if (a == "-r" || a == "--raw-count") o.canonical = 0;
        else if (a == "-H" || a == "--header") o.header = 1;
        else if (a == "-t" || a == "--threads") o.threads = atoi(val("--threads"));
        else if (a == "--device") o.device = atoi(val("--device"));
        else if (a == "--any-k") k_range_checked = false;  // superset: allow k outside 3..=7
        else if (a == "-p" || a == "--preset") {
            const std::string p = val("--preset");
            if (p == "csv") o.delim = ',';
            else if (p == "tsv") o.delim = '\t';
            else if (p == "spc") o.delim = ' ';
            else { fprintf(stderr, "error: invalid value '%s' for '--preset <PRESET>' [possible values: csv, tsv, spc]\n", p.c_str()); return 2; }
        } else if (a == "-h" || a == "--help") { usage(); return 0; }
        else { fprintf(stderr, "error: unexpected argument '%s' found\n", a.c_str()); usage(); return 2; }
    }
    if (in.empty() || out.empty()) {
        fprintf(stderr, "error: the following required arguments were not provided:\n%s%s", in.empty() ? "  --input <INPUT>\n" : "",
                out.empty() ? "  --output <OUTPUT>\n" : "");
        return 2;
    }
    if (k_range_checked && (o.k < 3 || o.k > 7)) {  // clap value_parser range(3..=7), args.rs:85
        fprintf(stderr, "error: invalid value '%d' for '--k-size <K_SIZE>': %d is not in 3..=7\n", o.k, o.k);
        return 2;
    }
    o.in_path = in.c_str();
    o.out_path = out.c_str();
    ktb_file_stats st{};
    const int rc = ktb_comp_oligo_file(&o, &st);
    if (rc != KTB_OK) {
        // the reference prints the error and still exits 0 (args.rs:260-262)
        fprintf(stderr, "Error: %s\n", ktb_last_error());
        return 0;
    }
    if (getenv("KTB_VERBOSE"))
        fprintf(stderr, "records %llu bases %llu written %llu B | parse %.1f ms gpu-wait %.1f ms write %.1f ms total %.1f ms\n",
                (unsigned long long)st.records, (unsigned long long)st.bases, (unsigned long long)st.bytes_written,
                st.parse_ms, st.gpu_wait_ms, st.write_ms, st.total_ms);
    return 0;
}
