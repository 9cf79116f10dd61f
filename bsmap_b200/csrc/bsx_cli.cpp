// bsx_cli.cpp -- the `bsmap` command line (main.cpp:234-476) over the C ABI.
//
// Same option grammar as mGetOptions (`-x val` and `-x=val`), same banner, same output files
// (SAM when -o ends in .sam, BSP otherwise; -2 for unpaired BSP hits).  Reads are parsed with the
// reference's token semantics (reads.cpp:83-146), mapped in large batches on the GPU, formatted on
// the host and written in input order (= the reference with -p 1, SURVEY.md App. A14).
// `-o x.bam` writes a coordinate-sorted BAM and its .bai in process (bsx_bam.cpp).
// Extensions: --methratio T and its --meth-* options pile methratio.py's table up on the device from the mapped batches,
// with the M-bias report (--meth-mbias, --meth-ignore), C/T SNP evidence (--meth-ct-snp) and the conversion filter
// (--meth-conversion-filter N, --meth-conversion-report FILE: drop alignments with N or more methylated non-CpG calls),
// and methylation levels per region and context reduced on the device (--meth-region-report FILE with --meth-regions BED
// or --meth-tiles W), and the proportion of discordant reads per CpG from the CpG calls of each alignment (--meth-pdr
// FILE, --meth-pdr-min-cpg K: the CpG calls an alignment needs to be scored, default 4), and the methylation patterns of
// the alignments over every window of four consecutive CpG sites, with methylation entropy and epipolymorphism
// (--meth-epialleles FILE), and the methylation haplotype load per region of --meth-regions or --meth-tiles
// (--meth-mhl FILE).
// Out of scope (errors out): SAM text input (broken in the reference too: it is opened as BAM), -q quality
// trimming, -M other than TC.
#include <cerrno>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <ctime>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <map>
#include <mutex>
#include <string>
#include <vector>
#include <sys/stat.h>
#include <unistd.h>
#include "bsx_internal.h"

namespace {

struct Opts {
    bsx_params p;
    std::string a, b, d, o, o2;
    unsigned read_start = 1, read_end = ~0u;
    int num_procs = 0, zero_qual = '!', qual_threshold = 0;   // -p: host threads (0 = all cores)
    std::string bam_out;         // -o x.bam: SAM text goes to a temporary file, then bsx_sam_to_sorted_bam (the reference: sam2bam.sh)
    std::string meth_out;        // --methratio FILE: methylation ratios straight from the device (no SAM needed)
    bsx_meth_opts mo;
    std::string meth_mbias;      // --meth-mbias FILE: the M-bias report of the same calls
    bool meth_ignore_set = false;
    int32_t meth_ignore[4] = {0, 0, 0, 0};   // --meth-ignore A,B,C,D: cycles dropped at the 5' / 3' ends of read 1 / read 2
    int meth_ct_snp = 0;                     // --meth-ct-snp MODE: BSX_CT_SNP_*
    int meth_conv = -1;                      // --meth-conversion-filter N (0..255); -1 = off
    std::string meth_conv_report;            // --meth-conversion-report FILE (alone: N = 0)
    std::string meth_region_report, meth_regions;   // --meth-region-report FILE, --meth-regions BED
    long long meth_tiles = 0;                // --meth-tiles W; 0 = none
    std::string meth_pdr;                    // --meth-pdr FILE
    int meth_pdr_min_cpg = 0;                // --meth-pdr-min-cpg K (1..255); 0 = not given (4); -1 = out of range
    std::string meth_epialleles;             // --meth-epialleles FILE
    std::string meth_mhl;                    // --meth-mhl FILE
    unsigned batch = 1u << 17;   // reads per GPU batch: small enough to keep the three host stages overlapped
    std::string gpus;            // -g: number of devices (default: all visible) or a comma list of device ids; output stays in input order
};

void usage() {
    printf("Usage:\tbsmap [options]\n"
           "       -a  <str>   query a file, FASTA/FASTQ format\n"
           "       -d  <str>   reference sequences file, FASTA format\n"
           "       -o  <str>   output alignment file, BSP/SAM format\n"
           "\n  Options for alignment:\n"
           "       -s  <int>   seed size, default=16(WGBS mode), 12(RRBS mode). min=8, max=16.\n"
           "       -v  <int>   maximum number of mismatches allowed on a read, <=15. default=2.\n"
           "       -w  <int>   maximum number of equal best hits to count, <=1000\n"
           "       -B  <int>   start from the Nth read or read pair, default: 1\n"
           "       -E  <int>   end at the Nth read or read pair, default: 4,294,967,295\n"
           "       -I  <int>   index interval, default=4\n"
           "       -p  <int>   number of host threads for parsing/formatting, default: all cores\n"
           "       -D  <str>   activating RRBS mapping mode and set restriction enzyme digestion sites, example: -D C-CGG\n"
           "       -S  <int>   seed for random number generation used in selecting multiple hits\n"
           "       -n  [0,1]   set mapping strand information. default: -n 0\n"
           "\n  Options for trimming:\n"
           "       -f  <int>   filter low-quality reads containing >n Ns, default=5\n"
           "       -A  <str>   3-end adapter sequence, default: none (no trim)\n"
           "       -L  <int>   map the first N nucleotides of the read, default:144 (map the whole read).\n"
           "\n  Options for reporting:\n"
           "       -r  [0,1]   how to report repeat hits, 0=none(unique hit/pair only); 1=random one, default:1.\n"
           "       -R          print corresponding reference sequences in SAM output, default=off\n"
           "       -u          report unmapped reads, default=off\n"
           "\n  Options for pair-end alignment:\n"
           "       -b  <str>   query b file\n"
           "       -m  <int>   minimal insert size allowed, default=28\n"
           "       -x  <int>   maximal insert size allowed, default=500\n"
           "       -2  <str>   output file of unpaired alignment hits\n"
           "       -h          help\n"
           "\n  Extensions (not in BSMAP 2.6):\n"
           "       -g  <int|list>  number of GPUs to map on (default: all visible) or a comma list of device ids; the index is\n"
           "                   replicated over NVLink, batches are dealt to the devices and written in input order\n"
           "       --methratio <str>   also write methratio.py's table, piled up on the GPU from the mapped batches\n"
           "                           (-o may then be omitted: no alignment text is produced at all)\n"
           "       --meth-unique --meth-pair --meth-zero --meth-cpg --meth-rmdup --meth-trim <int> --meth-min-depth <int>\n"
           "                           methratio.py's -u -p -z -g -r -t -m\n"
           "       --meth-mbias <str>  with --methratio: also write the M-bias report (methylation by read, context and cycle)\n"
           "       --meth-ignore <A,B,C,D>  with --methratio: drop calls in the first A / last B cycles of read 1 and the\n"
           "                           first C / last D cycles of read 2, from the table and the M-bias report\n"
           "       --meth-ct-snp <no-action|correct|skip>  with --methratio: count C/T SNP evidence from the opposite\n"
           "                           strand and write the table with eff_CT_count, rev_G_count and rev_GA_count\n"
           "       --meth-conversion-filter <int>  with --methratio: drop alignments with this many or more methylated\n"
           "                           non-CpG calls (incompletely converted reads), 0..255; 0 only counts them\n"
           "       --meth-conversion-report <str>  with --methratio: write the alignments by their number of methylated\n"
           "                           non-CpG calls (alone: --meth-conversion-filter 0)\n"
           "       --meth-region-report <str>  with --methratio: write methylation levels per region and context, over\n"
           "       --meth-regions <str>  the regions of a BED file (columns 1-3), or\n"
           "       --meth-tiles <int>  tiles of this many bases over every sequence\n"
           "       --meth-pdr <str>    with --methratio: write the proportion of discordant reads per CpG (alignments with\n"
           "                           both methylated and unmethylated CpG calls among those with enough CpG calls)\n"
           "       --meth-pdr-min-cpg <int>  with --meth-pdr: the CpG calls an alignment needs to count, 1..255 (default 4)\n"
           "       --meth-epialleles <str>  with --methratio: write the alignments' methylation patterns over every window of\n"
           "                           four consecutive CpG sites, with methylation entropy and epipolymorphism\n"
           "       --meth-mhl <str>    with --methratio and --meth-regions or --meth-tiles: write the methylation haplotype\n"
           "                           load (MHL, uMHL) per region\n\n");
    exit(1);
}

void set_digestion(Opts &o, const char *a) {   // Param::SetDigestionSite (param.cpp:95-106)
    std::string s = a;
    size_t pos = s.find('-');
    if (pos == std::string::npos) { printf("Digestion position not marked, use '-' to mark. example: 'C-CGG'\n"); exit(1); }
    s.erase(pos, 1);
    memset(o.p.digest_site, 0, sizeof o.p.digest_site);
    strncpy(o.p.digest_site, s.c_str(), sizeof o.p.digest_site - 1);
    o.p.digest_pos = (int)pos; o.p.rrbs = 1; o.p.index_interval = 1; o.p.seed_size = 12;
}

// mGetOptions (main.cpp:234-289); returns the argv index of an unknown option, 0 when fine
int get_options(int argc, char **argv, Opts &o) {
    for (int i = 1; i < argc; i++) {
        if (argv[i][0] != '-') return i;
        if (argv[i][1] == '-') {
            // extensions (the reference's parser stops at any of these): methratio.py's table from the device-side
            // pile-up, --methratio FILE [--meth-unique --meth-pair --meth-zero --meth-cpg --meth-trim N --meth-min-depth N]
            const std::string a = argv[i] + 2;
            if (a == "methratio" && i + 1 < argc) o.meth_out = argv[++i];
            else if (a == "meth-unique") o.mo.unique = 1;
            else if (a == "meth-pair") o.mo.pair = 1;
            else if (a == "meth-zero") o.mo.meth0 = 1;
            else if (a == "meth-cpg") o.mo.combine_cpg = 1;
            else if (a == "meth-rmdup") o.mo.rm_dup = 1;
            else if (a == "meth-trim" && i + 1 < argc) o.mo.trim_fillin = atoi(argv[++i]);
            else if (a == "meth-min-depth" && i + 1 < argc) o.mo.min_depth = atoi(argv[++i]);
            else if (a == "meth-mbias" && i + 1 < argc) o.meth_mbias = argv[++i];
            else if (a == "meth-ignore" && i + 1 < argc) {
                const char *q = argv[++i];
                for (int k = 0; k < 4; k++) {
                    char *e; const long x = strtol(q, &e, 10);
                    if (e == q || x < 0 || x > 0x7fffffff || *e != (k < 3 ? ',' : '\0')) return i;   // "unknown option: <value>"
                    o.meth_ignore[k] = (int32_t)x; q = e + 1;
                }
                o.meth_ignore_set = true;
            }
            else if (a == "meth-ct-snp" && i + 1 < argc) {
                o.meth_ct_snp = bsx_ct_snp_mode(argv[++i]);
                if (!o.meth_ct_snp) return i;                                                            // "unknown option: <value>"
            }
            else if (a == "meth-conversion-filter" && i + 1 < argc) {
                const char *v = argv[++i]; char *e; const long x = strtol(v, &e, 10);
                if (*e || e == v || x < 0 || x > BSX_CONV_BINS - 1) return i;                             // "unknown option: <value>"
                o.meth_conv = (int)x;
            }
            else if (a == "meth-conversion-report" && i + 1 < argc) o.meth_conv_report = argv[++i];
            else if (a == "meth-region-report" && i + 1 < argc) o.meth_region_report = argv[++i];
            else if (a == "meth-regions" && i + 1 < argc) o.meth_regions = argv[++i];
            else if (a == "meth-tiles" && i + 1 < argc) {
                const char *v = argv[++i]; char *e; const long long x = strtoll(v, &e, 10);
                if (*e || e == v || x < 1) return i;                                                      // "unknown option: <value>"
                o.meth_tiles = x;
            }
            else if (a == "meth-pdr" && i + 1 < argc) o.meth_pdr = argv[++i];
            else if (a == "meth-epialleles" && i + 1 < argc) o.meth_epialleles = argv[++i];
            else if (a == "meth-mhl" && i + 1 < argc) o.meth_mhl = argv[++i];
            else if (a == "meth-pdr-min-cpg" && i + 1 < argc) {
                const char *v = argv[++i]; char *e; const long x = strtol(v, &e, 10);
                o.meth_pdr_min_cpg = (*e || e == v || x < 1 || x > 255) ? -1 : (int)x;
            }
            else return i;
            continue;
        }
        const char c = argv[i][1];
        const char *val = nullptr;
        const bool flag = (c == 'R' || c == 'u' || c == 'h');
        if (c == 0 || !strchr("abdo2smxnrIvwqfzpARuBEDMLShg", c)) return i;   // default: return i (main.cpp:283)
        if (!flag) {
            if (argv[i][2] == 0) { if (i + 1 >= argc) return i; val = argv[++i]; }
            else if (argv[i][2] == '=') val = argv[i] + 3;
            else return i;
        } else if (argv[i][2] != 0) return i;
        switch (c) {
            case 'a': o.a = val; break;
            case 'b': o.b = val; o.p.pairend = 1; break;
            case 'd': o.d = val; break;
            case 'o': o.o = val; break;
            case '2': o.o2 = val; break;
            case 's': o.p.seed_size = atoi(val); if (o.p.rrbs) o.p.seed_size = 12; break;
            case 'm': o.p.min_insert = atoi(val); break;
            case 'x': o.p.max_insert = atoi(val); break;
            case 'n': o.p.chains = atoi(val) != 0; break;
            case 'r': o.p.report_repeat_hits = atoi(val); break;
            case 'I': o.p.index_interval = atoi(val); if (o.p.rrbs) o.p.index_interval = 1;
                      if (o.p.index_interval > 16) { fprintf(stderr, "index interval exceeds max value:16\n"); exit(1); } break;
            case 'v': o.p.max_snp_num = atoi(val); if (o.p.max_snp_num > BSX_MAXSNPS) { fprintf(stderr, "number of mismatches exceeds max value:%d\n", BSX_MAXSNPS); exit(1); } break;
            case 'w': o.p.max_num_hits = atoi(val); if (o.p.max_num_hits > BSX_MAXHITS) { fprintf(stderr, "number of multi-hits exceeds max value:%d\n", BSX_MAXHITS); exit(1); } break;
            case 'q': o.qual_threshold = atoi(val); break;
            case 'f': o.p.max_ns = atoi(val); break;
            case 'z': o.zero_qual = atoi(val); break;
            case 'p': o.num_procs = atoi(val); break;
            case 'A': if (o.p.n_adapter < BSX_MAX_ADAPTERS) { strncpy(o.p.adapter[o.p.n_adapter], val, 63); o.p.n_adapter++; } break;
            case 'R': o.p.out_ref = 1; break;
            case 'u': o.p.out_unmap = 1; break;
            case 'B': { int v = atoi(val); o.read_start = v > 1 ? (unsigned)v : 1u; } break;
            case 'E': o.read_end = (unsigned)atoi(val); break;
            case 'D': set_digestion(o, val); break;
            case 'M': if (!((val[0] == 'T' || val[0] == 't') && (val[1] == 'C' || val[1] == 'c'))) { fprintf(stderr, "-M %s: only the TC transition is supported by the GPU path\n", val); exit(1); } break;
            case 'L': o.p.max_readlen = atoi(val); break;
            case 'S': o.p.randseed = atoi(val); break;
            case 'g': o.gpus = val; break;
            case 'h': usage(); break;
            default: return i;
        }
    }
    return 0;
}

// bounded hand-off between pipeline stages
template <class T> struct Chan {
    std::mutex m; std::condition_variable cv; std::vector<T> q; size_t cap; bool closed = false;
    explicit Chan(size_t c) : cap(c) {}
    void push(T &&v) { std::unique_lock<std::mutex> l(m); cv.wait(l, [&] { return q.size() < cap; }); q.push_back(std::move(v)); cv.notify_all(); }
    bool pop(T &v) { std::unique_lock<std::mutex> l(m); cv.wait(l, [&] { return !q.empty() || closed; }); if (q.empty()) return false; v = std::move(q.front()); q.erase(q.begin()); cv.notify_all(); return true; }
    void close() { std::unique_lock<std::mutex> l(m); closed = true; cv.notify_all(); }
    // non-blocking forms (recycling pools: an empty pool means "make a new one", a full pool "drop it")
    bool try_push(T &&v) { std::unique_lock<std::mutex> l(m); if (q.size() >= cap) return false; q.push_back(std::move(v)); cv.notify_all(); return true; }
    bool try_pop(T &v) { std::unique_lock<std::mutex> l(m); if (q.empty()) return false; v = std::move(q.back()); q.pop_back(); return true; }
};

// hand-off that releases items in sequence order whatever order they arrive in (several mapper threads, one formatter)
template <class T> struct Ordered {
    std::mutex m; std::condition_variable cv; std::map<unsigned, T> q; unsigned next = 0; bool closed = false;
    void push(unsigned seq, T &&v) { std::unique_lock<std::mutex> l(m); q.emplace(seq, std::move(v)); cv.notify_all(); }
    bool pop(T &v) {
        std::unique_lock<std::mutex> l(m);
        cv.wait(l, [&] { return (!q.empty() && q.begin()->first == next) || closed; });
        if (q.empty() || q.begin()->first != next) return false;
        v = std::move(q.begin()->second); q.erase(q.begin()); next++;
        return true;
    }
    void close() { std::unique_lock<std::mutex> l(m); closed = true; cv.notify_all(); }
};
// free list of pinned staging slots: taken by the cutter, returned by the formatter
struct SlotPool {
    std::mutex m; std::condition_variable cv; std::vector<int> free_;
    void put(int s) { std::unique_lock<std::mutex> l(m); free_.push_back(s); cv.notify_all(); }
    int take() { std::unique_lock<std::mutex> l(m); cv.wait(l, [&] { return !free_.empty(); }); const int s = free_.back(); free_.pop_back(); return s; }
};

struct Views { std::vector<bsx_view> name, seq, qual; std::vector<std::string> store; std::vector<std::shared_ptr<std::vector<char>>> keep; };
// the batch's views leave the reader: with them the strings and the stream windows they point into
void take_views(bsx_reads *r, Views &v) { v.name.swap(r->name); v.seq.swap(r->seq); v.qual.swap(r->qual); v.store.swap(r->slow_store); v.keep.swap(r->keep); }

struct Job { uint32_t n = 0; int slot = 0; unsigned done_index = 0; Views a, b; };
struct Text { std::vector<std::string> main, unpair; unsigned done_index = 0; };

template <class T> T *pinned(size_t count) {
    void *p = nullptr;
    if (cudaHostAlloc(&p, count * sizeof(T), cudaHostAllocDefault) != cudaSuccess) { fprintf(stderr, "cudaHostAlloc of %zu bytes failed\n", count * sizeof(T)); exit(1); }
    return (T *)p;
}

// The chunks of one batch, written where they belong in the file by a few threads at once (pwrite at precomputed
// offsets; BSX_CLI_WRITE_THREADS, default 4).  Buffered writes to one file serialise in the kernel: on the GPU box the stage
// takes 1.2 s for 5.5 GB of SAM (4.6 GB/s) with 2, 4, 8 or 16 writers alike -- it is the limit of the map loop.
// Streams that cannot seek (pipes, /dev/stdout) get the chunks in order through write().
struct OutFile {
    int fd = -1; off_t off = 0; bool seekable = false;
    void open(FILE *f) { fflush(f); fd = fileno(f); off = lseek(fd, 0, SEEK_CUR); seekable = off >= 0; struct stat st; if (seekable && (fstat(fd, &st) != 0 || !S_ISREG(st.st_mode))) seekable = false; }
    bool write_chunks(const std::vector<std::string> &chunks, int threads) {
        std::atomic<int> bad{0};
        auto put = [&](const std::string &c, off_t at, bool positional) {
            size_t done = 0;
            while (done < c.size()) {
                const ssize_t w = positional ? pwrite(fd, c.data() + done, c.size() - done, at + (off_t)done) : write(fd, c.data() + done, c.size() - done);
                if (w <= 0) { if (w < 0 && errno == EINTR) continue; bad = 1; return; }
                done += (size_t)w;
            }
        };
        if (!seekable) { for (const std::string &c : chunks) put(c, 0, false); return !bad; }
        std::vector<off_t> at(chunks.size() + 1, off);
        for (size_t k = 0; k < chunks.size(); k++) at[k + 1] = at[k] + (off_t)chunks[k].size();
        static const int wt = [] { const char *e = getenv("BSX_CLI_WRITE_THREADS"); const int v = e ? atoi(e) : 0; return v > 0 ? v : 4; }();
        bsx_parallel(std::min<int>(threads, wt), chunks.size(), [&](int, size_t b, size_t e) { for (size_t k = b; k < e; k++) put(chunks[k], at[k], true); });
        off = at[chunks.size()];
        return !bad;
    }
};

double now() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }
bool g_exit_after_main = false;

// -g: "" = every visible device, "N" = the first N, "a,b,c" = these device ids (an id may repeat: several mappers on one GPU)
std::vector<int> device_list(const std::string &g) {
    const int have = std::max(1, bsx_device_count());
    std::vector<int> d;
    if (g.find(',') != std::string::npos) {
        size_t q = 0;
        while (q <= g.size()) {
            const size_t e = g.find(',', q);
            const std::string t = g.substr(q, e == std::string::npos ? std::string::npos : e - q);
            if (!t.empty()) { const int v = atoi(t.c_str()); if (v < 0 || v >= have) { fprintf(stderr, "-g: no device %d (have %d)\n", v, have); exit(1); } d.push_back(v); }
            if (e == std::string::npos) break;
            q = e + 1;
        }
    } else {
        int n = g.empty() ? have : atoi(g.c_str());
        if (n < 1 || n > have) n = have;
        for (int i = 0; i < n; i++) d.push_back(i);
    }
    if (d.empty()) d.push_back(0);
    return d;
}

}  // namespace

extern "C" int bsx_cli_main(int argc, char **argv) {
    const time_t t0 = time(nullptr);
    const double t_start = now();
    printf("\nBSMAP v2.6 (bsmap_b200: B200-native hot path)\n");
    if (argc == 1) usage();
    { time_t t = time(nullptr); printf("Start at:  %s\n", ctime(&t)); }
    Opts o; bsx_params_default(&o.p); bsx_meth_opts_default(&o.mo);
    if (int bad = get_options(argc, argv, o)) { printf("unknown option: %s\n", argv[bad]); exit(bad); }
    if (o.meth_out.empty() && (!o.meth_mbias.empty() || o.meth_ignore_set)) { fprintf(stderr, "--meth-mbias and --meth-ignore need --methratio\n"); return 1; }
    if (o.meth_out.empty() && o.meth_ct_snp) { fprintf(stderr, "--meth-ct-snp needs --methratio\n"); return 1; }
    if (o.meth_out.empty() && (o.meth_conv >= 0 || !o.meth_conv_report.empty())) {
        fprintf(stderr, "--meth-conversion-filter and --meth-conversion-report need --methratio\n"); return 1; }
    if (!o.meth_conv_report.empty() && o.meth_conv < 0) o.meth_conv = 0;
    if (o.meth_out.empty() && !o.meth_mhl.empty()) { fprintf(stderr, "--meth-mhl needs --methratio\n"); return 2; }
    if (!o.meth_mhl.empty() && o.meth_regions.empty() && !o.meth_tiles) { fprintf(stderr, "--meth-mhl needs --meth-regions BED or --meth-tiles W\n"); return 2; }
    const bool region_opts = !o.meth_region_report.empty() || !o.meth_regions.empty() || o.meth_tiles;
    if (o.meth_out.empty() && region_opts) { fprintf(stderr, "--meth-region-report, --meth-regions and --meth-tiles need --methratio\n"); return 1; }
    if (!o.meth_regions.empty() && o.meth_tiles) { fprintf(stderr, "--meth-regions and --meth-tiles exclude each other\n"); return 1; }
    if (region_opts && o.meth_region_report.empty() && o.meth_mhl.empty()) {
        fprintf(stderr, "--meth-regions / --meth-tiles need --meth-region-report FILE or --meth-mhl FILE\n"); return 1; }
    if (!o.meth_region_report.empty() && o.meth_regions.empty() && !o.meth_tiles) { fprintf(stderr, "--meth-region-report needs --meth-regions BED or --meth-tiles W\n"); return 1; }
    if (o.meth_pdr_min_cpg < 0) { fprintf(stderr, "--meth-pdr-min-cpg: expected an integer 1..255\n"); return 2; }
    if (o.meth_pdr_min_cpg && o.meth_pdr.empty()) { fprintf(stderr, "--meth-pdr-min-cpg needs --meth-pdr FILE\n"); return 2; }
    if (o.meth_out.empty() && !o.meth_pdr.empty()) { fprintf(stderr, "--meth-pdr needs --methratio\n"); return 2; }
    if (!o.meth_pdr.empty() && !o.meth_pdr_min_cpg) o.meth_pdr_min_cpg = 4;
    if (o.meth_out.empty() && !o.meth_epialleles.empty()) { fprintf(stderr, "--meth-epialleles needs --methratio\n"); return 2; }
    if (o.qual_threshold != 0) { fprintf(stderr, "-q quality trimming is not supported by the GPU path\n"); return 1; }
    if (o.o.size() > 4) {
        if (o.o.compare(o.o.size() - 4, 4, ".sam") == 0) o.p.out_sam = 1;
        else if (o.o.compare(o.o.size() - 4, 4, ".bam") == 0) { o.p.out_sam = 1; o.bam_out = o.o; o.o += ".sam.tmp"; }   // param.out_sam = 2 (main.cpp:295)
    }
    // the CUDA context comes up on its own thread while this one parses the reference FASTA
    bsx_index *ix = nullptr;
    std::thread ctx_thread([&o] { cudaSetDevice(device_list(o.gpus)[0]); cudaFree(nullptr); });
    std::vector<std::string> ref_names, ref_seqs;
    // BSX_REF_CACHE=<dir>: keep the packed reference of every FASTA seen there (keyed by name, size and mtime);
    // the next run skips the FASTA parse and rebuilds the seed table from the packed strand on the device
    std::string cache_path;
    if (const char *dir = getenv("BSX_REF_CACHE")) {
        struct stat st;
        if (*dir && !o.p.rrbs && o.meth_out.empty() && stat(o.d.c_str(), &st) == 0) {
            const size_t sl = o.d.find_last_of('/');
            cache_path = std::string(dir) + "/" + (sl == std::string::npos ? o.d : o.d.substr(sl + 1)) + "." + std::to_string((long long)st.st_size) +
                         "." + std::to_string((long long)st.st_mtime) + ".bsxpack";
        }
    }
    bool from_cache = !cache_path.empty() && access(cache_path.c_str(), R_OK) == 0;
    int lrc = BSX_OK;
    if (!from_cache) lrc = bsx_load_fasta(o.d.c_str(), ref_names, ref_seqs);
    const double t_fa = now();
    ctx_thread.join();
    const double t_ctx = now();
    const int dev0 = device_list(o.gpus)[0];
    if (from_cache && bsx_index_create_from_packed(&o.p, cache_path.c_str(), dev0, &ix) != BSX_OK) {
        fprintf(stderr, "warning: %s -- falling back to %s\n", bsx_last_error(), o.d.c_str());
        from_cache = false; ix = nullptr;
        lrc = bsx_load_fasta(o.d.c_str(), ref_names, ref_seqs);
    }
    if (lrc != BSX_OK) { fprintf(stderr, "%s\n", bsx_last_error()); return 1; }
    if (!from_cache) {
        std::vector<const char *> np, sp; std::vector<uint32_t> ln;
        for (size_t k = 0; k < ref_seqs.size(); k++) { np.push_back(ref_names[k].c_str()); sp.push_back(ref_seqs[k].data()); ln.push_back((uint32_t)ref_seqs[k].size()); }
        if (bsx_index_create(&o.p, (int)ref_seqs.size(), np.data(), sp.data(), ln.data(), dev0, &ix) != BSX_OK) { fprintf(stderr, "%s\n", bsx_last_error()); return 1; }
        if (!cache_path.empty() && bsx_index_save_packed(ix, cache_path.c_str()) != BSX_OK) fprintf(stderr, "warning: %s\n", bsx_last_error());
    }
    if (o.meth_out.empty()) std::vector<std::string>().swap(ref_seqs);   // the methratio report prints reference context
    bsx_regions regions;                                                 // read before mapping, so that a bad BED fails early
    if ((!o.meth_regions.empty() && bsx_regions_bed(ix, nullptr, o.meth_regions.c_str(), regions) != BSX_OK) ||
        (o.meth_tiles && bsx_regions_tiles(ix, nullptr, (uint64_t)o.meth_tiles, regions) != BSX_OK)) {
        fprintf(stderr, "%s\n", bsx_last_error()); return 1; }
    bsx_index_info info; bsx_index_get_info(ix, &info);
    unsigned long long sum_len = 0; for (uint32_t k = 0; k < info.n_seq; k++) sum_len += bsx_index_seq_size(ix, k);
    printf("Load in %u db seqs, total size %llu bp. %ld secs passed\n", info.n_seq, sum_len, (long)(time(nullptr) - t0));
    printf("total_kmers: %llu\n", (unsigned long long)info.n_keys);
    printf("Create seed table. %ld secs passed\n", (long)(time(nullptr) - t0));

    const bsx_params &p = o.p;
    printf("max mismatches: %d\tmax multi-hits: %d\tmax Ns: %d\tseed size: %d\tindex interval: %d\n", p.max_snp_num, p.max_num_hits, p.max_ns, p.seed_size, p.index_interval);
    printf("quality cutoff: %d\tbase quality char: '%c'\n", o.qual_threshold, o.zero_qual);
    printf("min fragment size:%d\tmax fragemt size:%d\n", p.min_insert, p.max_insert);
    printf("start from read #%u\tend at read #%u\n", o.read_start, o.read_end);
    printf("additional alignment: T in reads => C in reference\n");
    printf("param.chains:%d\n", p.chains);
    if (p.pairend) { printf("mapping strand (read_1): ++,-+%s\n", p.chains ? ",+-,--" : ""); printf("mapping strand (read_2): +-,--%s\n", p.chains ? ",++,-+" : ""); }
    else printf("mapping strand: ++,-+%s\n", p.chains ? ",+-,--" : "");
    for (int i = 0; i < p.n_adapter; i++) printf("adapter sequence%d: %s\n", i + 1, p.adapter[i]);
    if (p.rrbs) { std::string s = p.digest_site; printf("RRBS mode. digestion site: %s-%s\n", s.substr(0, p.digest_pos).c_str(), s.substr(p.digest_pos).c_str()); }

    const bool pe = !o.a.empty() && !o.b.empty();
    if (o.a.empty()) { fprintf(stderr, "missing query file(s)\n"); return 1; }
    const bool timing = getenv("BSX_CLI_TIMING") != nullptr;
    const double t_idx = now();
    bsx_reads *ra = nullptr, *rb = nullptr;
    int rc = bsx_reads_open(o.a.c_str(), o.zero_qual, p.max_readlen, &ra);
    if (rc == BSX_ERR_IO) { fprintf(stderr, "failed to open read file%s (check -a option): %s\n", pe ? " #1" : "", o.a.c_str()); return 1; }
    if (rc == BSX_OK && pe) {
        rc = bsx_reads_open(o.b.c_str(), o.zero_qual, p.max_readlen, &rb);
        if (rc == BSX_ERR_IO) { fprintf(stderr, "failed to open read file #2 (check -b option): %s\n", o.b.c_str()); return 1; }
    }
    if (rc != BSX_OK) { fprintf(stderr, "fatal error: unrecognizable format of reads file (FASTA, FASTQ, gzip of either, or BAM).\n"); return 1; }
    if (pe) { bsx_reads_set_readset(ra, 1); bsx_reads_set_readset(rb, 2); }
    if (pe) printf("Pair-end alignment(GPU)\nQuery: %s  %s  Reference: %s  Output: %s  %s\n", o.a.c_str(), o.b.c_str(), o.d.c_str(), o.o.c_str(), o.o2.c_str());
    else printf("Single read alignment(GPU)\nQuery: %s  Reference: %s  Output: %s\n", o.a.c_str(), o.d.c_str(), o.o.c_str());
    const bool no_text = o.o.empty() && !o.meth_out.empty();             // --methratio without -o: no alignment text at all
    FILE *fout = fopen(no_text ? "/dev/null" : o.o.c_str(), "wb");
    if (!fout) { fprintf(stderr, "failed to open output file (check -o option): %s\n", o.o.c_str()); return 1; }
    FILE *fun = nullptr;
    if (pe && !p.out_sam && !no_text) { fun = fopen(o.o2.c_str(), "wb"); if (!fun) { fprintf(stderr, "failed to open output file for unpaired hits (check -2 option): %s\n", o.o2.c_str()); return 1; } }
    if (p.out_sam && !no_text) { std::vector<char> text; size_t n = bsx_format_header(ix, nullptr, 0); text.resize(n + 1); bsx_format_header(ix, text.data(), n + 1); fwrite(text.data(), 1, n, fout); fflush(fout); }

    const unsigned stride = 160;
    const int threads = bsx_host_threads(o.num_procs);
    if (const char *e = getenv("BSX_CLI_BATCH")) { const int v = atoi(e); if (v > 0) o.batch = (unsigned)v; }
    // devices: -g N (default all visible).  Device 0 holds the index and starts mapping at once; the others come up on
    // their own threads (context, replica of the index over NVLink, mapper) and join the pool when ready, so a small
    // input never waits for them.  --methratio piles up on one device.
    std::vector<int> devs = device_list(o.gpus);
    if (!o.meth_out.empty()) devs.resize(1);
    const int n_dev = (int)devs.size();
    std::vector<bsx_mapper *> mps((size_t)n_dev, nullptr);
    std::vector<bsx_index *> ixs((size_t)n_dev, nullptr);
    ixs[0] = ix;
    if (bsx_mapper_create(ix, &p, o.batch, stride, &mps[0]) != BSX_OK) { fprintf(stderr, "%s\n", bsx_last_error()); return 1; }
    bsx_mapper *mp = mps[0];
    bsx_meth *mh = nullptr;
    if (!o.meth_out.empty()) {
        // SAM rules (mate-overlap removal) unless the alignment output is BSP: the table then equals methratio.py run on -o
        if (bsx_meth_create(ix, &mh) != BSX_OK || (!o.meth_mbias.empty() && bsx_meth_enable_mbias(mh) != BSX_OK) ||
            (o.meth_ignore_set && bsx_meth_set_ignore(mh, o.meth_ignore) != BSX_OK) ||
            (o.meth_ct_snp && bsx_meth_enable_ct_snp(mh, o.meth_ct_snp) != BSX_OK) ||
            (o.meth_conv >= 0 && bsx_meth_enable_conversion_filter(mh, o.meth_conv) != BSX_OK) ||
            (!o.meth_pdr.empty() && bsx_meth_enable_pdr(mh, o.meth_pdr_min_cpg) != BSX_OK) ||
            (!o.meth_epialleles.empty() && bsx_meth_enable_epialleles(mh) != BSX_OK) ||
            (!o.meth_mhl.empty() && bsx_meth_enable_mhl(mh) != BSX_OK) ||
            bsx_mapper_attach_meth(mp, mh, &o.mo, (p.out_sam || no_text) ? 1 : 0) != BSX_OK) {
            fprintf(stderr, "%s\n", bsx_last_error()); return 1; }
    }
    bsx_reads_skip(ra, o.read_start - 1); if (pe) bsx_reads_skip(rb, o.read_start - 1);
    unsigned index_a = o.read_start - 1;
    // pinned staging slots (upload buffers + result records), handed round by a free list: a slot is taken by the cutter,
    // travels with its batch through a mapper thread and the formatter, and comes back when its text exists
    const int NSLOT = 2 * n_dev + 2;
    std::vector<char *> sa(NSLOT), sb(NSLOT); std::vector<uint16_t *> la(NSLOT), lb(NSLOT);
    std::vector<bsx_rec *> reca(NSLOT), recb(NSLOT); std::vector<bsx_pair_rec *> recp(NSLOT); std::vector<uint16_t *> cnta(NSLOT), cntb(NSLOT);
    const bool want_counts = !p.out_sam;   // per-level hit counts are a BSP column
    SlotPool pool;
    for (int k = 0; k < NSLOT; k++) {
        sa[k] = pinned<char>((size_t)o.batch * stride); la[k] = pinned<uint16_t>(o.batch);
        sb[k] = pe ? pinned<char>((size_t)o.batch * stride) : nullptr; lb[k] = pe ? pinned<uint16_t>(o.batch) : nullptr;
        reca[k] = pinned<bsx_rec>(o.batch); cnta[k] = want_counts ? pinned<uint16_t>((size_t)o.batch * 16) : nullptr;
        recb[k] = pe ? pinned<bsx_rec>(o.batch) : nullptr; recp[k] = pe ? pinned<bsx_pair_rec>(o.batch) : nullptr;
        cntb[k] = pe && want_counts ? pinned<uint16_t>((size_t)o.batch * 16) : nullptr;
        pool.put(k);
    }
    unsigned long long n_aligned = 0, n_pairs = 0, n_a = 0, n_b = 0;
    double t_parse = 0, t_fmt = 0, t_write = 0;
    std::vector<double> t_map((size_t)n_dev, 0.0); std::vector<unsigned long long> n_map((size_t)n_dev, 0);
    Ordered<Job> jobs; Chan<Text> texts(2);
    Chan<Text> spare(4);
    Chan<Views> spare_views(8);                     // view arrays of formatted batches go back to the cutter with their capacity                            // written texts come back with their buffers: the formatter fills them again (no fresh pages)
    std::atomic<int> fail{0};
    const double t_alloc = now();
    std::thread formatter([&] {
        Job j;
        while (jobs.pop(j)) {
            const double t = now();
            Text tx;
            spare.try_pop(tx);
            tx.done_index = j.done_index;
            if (no_text) {   // counts only (the rules of s_OutHit / s_OutHitPair / s_OutHitUnpair for "printed as mapped")
                auto mapped = [&](const bsx_rec &r) { const int n = r.status ? -1 : (int)r.nhits; return n >= 1 && !(n > 1 && p.report_repeat_hits == 0); };
                for (uint32_t t = 0; t < j.n; t++) {
                    if (!pe) n_aligned += mapped(reca[j.slot][t]);
                    else if (recp[j.slot][t].paired) n_pairs++;
                    else { n_a += mapped(reca[j.slot][t]); n_b += mapped(recb[j.slot][t]); }
                }
            } else if (!pe) {
                uint32_t na = 0;
                bsx_format_se_chunks(ix, &p, j.n, j.a.name.data(), j.a.seq.data(), j.a.qual.data(), 0, reca[j.slot], cnta[j.slot], threads, tx.main, &na);
                n_aligned += na;
            } else {
                uint32_t st[3] = {0, 0, 0};
                bsx_format_pe_chunks(ix, &p, j.n, j.a.name.data(), j.a.seq.data(), j.a.qual.data(), j.b.name.data(), j.b.seq.data(), j.b.qual.data(),
                                     recp[j.slot], reca[j.slot], recb[j.slot], cnta[j.slot], cntb[j.slot], threads, tx.main, tx.unpair, st);
                n_pairs += st[0]; n_a += st[1]; n_b += st[2];
            }
            pool.put(j.slot);
            j.a.keep.clear(); j.a.store.clear(); spare_views.try_push(std::move(j.a));   // the stream windows and token strings are released here
            if (pe) { j.b.keep.clear(); j.b.store.clear(); spare_views.try_push(std::move(j.b)); }
            t_fmt += now() - t;
            texts.push(std::move(tx));
        }
        texts.close();
    });
    OutFile of_main, of_un;
    of_main.open(fout); if (fun) of_un.open(fun);
    std::thread writer([&] {
        Text tx;
        while (texts.pop(tx)) {
            const double t = now();
            if (!of_main.write_chunks(tx.main, threads)) fail = 2;
            if (fun && !of_un.write_chunks(tx.unpair, threads)) fail = 2;
            t_write += now() - t;
            printf("%u reads finished. %ld secs passed\n", tx.done_index, (long)(time(nullptr) - t0));
            spare.try_push(std::move(tx));
        }
    });
    // cut (this thread) || map (one thread per device) || format || write
    struct CutJob { uint32_t n = 0; unsigned first = 0, done_index = 0, seq = 0; int slot = 0; Views a, b; };
    Chan<CutJob> cuts((size_t)n_dev);
    std::vector<std::thread> mappers;
    std::atomic<int> dev_up{0};
    for (int g = 0; g < n_dev; g++) mappers.emplace_back([&, g] {
        if (g > 0) {   // bring the device up: context, replica of the index (cudaMemcpyPeer over NVLink), mapper
            if (bsx_index_replicate(ix, devs[g], &ixs[g]) != BSX_OK || bsx_mapper_create(ixs[g], &p, o.batch, stride, &mps[g]) != BSX_OK) {
                fprintf(stderr, "warning: device %d not used: %s\n", devs[g], bsx_last_error());
                dev_up++;
                return;                                             // the other devices carry on
            }
        }
        dev_up++;
        CutJob c;
        while (cuts.pop(c)) {
            Job j; j.n = c.n; j.slot = c.slot; j.done_index = c.done_index;
            if (!fail) {
                const double t = now();
                const int s = c.slot;
                int mrc;
                if (!pe) mrc = bsx_map_se(mps[g], c.n, sa[s], la[s], c.first, 0, reca[s], cnta[s]);
                else mrc = bsx_map_pe(mps[g], c.n, sa[s], la[s], sb[s], lb[s], c.first, recp[s], reca[s], recb[s], cnta[s], cntb[s]);
                t_map[g] += now() - t; n_map[g] += c.n;
                if (mrc != BSX_OK) { fprintf(stderr, "%s\n", bsx_last_error()); fail = 1; }
            }
            if (fail) j.n = 0;                                      // keep the sequence flowing so that nobody blocks
            j.a = std::move(c.a); j.b = std::move(c.b);
            jobs.push(c.seq, std::move(j));
        }
    });
    // BSX_CLI_WAIT_DEVICES=1: do not start before every device is up (reproducible multi-GPU timings and tests)
    if (getenv("BSX_CLI_WAIT_DEVICES")) while (dev_up.load() < n_dev) usleep(200);
    for (unsigned k = 0; !fail; k++) {
        const unsigned first = index_a;
        const unsigned want = (unsigned)std::min<unsigned long long>(o.batch, index_a < o.read_end ? (unsigned long long)o.read_end - index_a : 0);
        if (!want) break;
        const int slot = pool.take();
        const double t = now();
        const unsigned n1 = bsx_reads_next(ra, want, stride, sa[slot], la[slot], threads);
        const unsigned n2 = pe ? bsx_reads_next(rb, want, stride, sb[slot], lb[slot], threads) : n1;
        t_parse += now() - t;
        if (!n1 || n1 != n2) break;
        index_a += n1;
        CutJob c; c.n = n1; c.first = first; c.slot = slot; c.seq = k; c.done_index = index_a - o.read_start + 1;
        spare_views.try_pop(c.a); if (pe) spare_views.try_pop(c.b);          // recycled arrays, swapped into the readers for the next batch
        take_views(ra, c.a); if (pe) take_views(rb, c.b);
        cuts.push(std::move(c));
    }
    cuts.close();
    bool input_failed = false;
    if (bsx_reads_failed(ra) || (pe && bsx_reads_failed(rb))) {   // a corrupt / truncated gzip input: what was read is mapped and written, the run fails
        fprintf(stderr, "error: %s\n", bsx_last_error());
        input_failed = true;
    }
    for (auto &t : mappers) t.join();
    jobs.close();
    const double t_loop = now();
    formatter.join(); writer.join();
    if (fclose(fout) != 0) fail = 2;
    if (fun && fclose(fun) != 0) fail = 2;
    if (fail == 2) fprintf(stderr, "error: writing the alignment output failed (disk full?)%s\n", o.bam_out.empty() ? "" : "; the BAM conversion is skipped");
    const double t_drain = now();
    if (timing) fprintf(stderr, "[bsx timing] wall: reference FASTA %.3f s || CUDA context (ready at %.3f s), index %.3f s, buffers+mapper %.3f s, map loop %.3f s, drain %.3f s | stage busy time: cut %.3f s, map %.3f s, format %.3f s, write %.3f s | reads cut by line %llu, by token reader %llu | %d host threads\n",
                        t_fa - t_start, t_ctx - t_start, t_idx - t_ctx, t_alloc - t_idx, t_loop - t_alloc, t_drain - t_loop, t_parse, t_map[0], t_fmt, t_write, (unsigned long long)(ra->n_fast + (rb ? rb->n_fast : 0)),
                        (unsigned long long)(ra->n_slow + (rb ? rb->n_slow : 0)), threads);
    if (timing && n_dev > 1) for (int g = 0; g < n_dev; g++) fprintf(stderr, "[bsx timing] device %d: %llu reads in %.3f s of map calls\n", devs[g], n_map[g], t_map[g]);
    bsx_reads_close(ra); bsx_reads_close(rb);
    if (fail || input_failed) return 1;
    if (mh) {
        const double t = now();
        std::vector<const char *> sp; std::vector<uint32_t> ln;
        for (size_t k = 0; k < ref_seqs.size(); k++) { sp.push_back(ref_seqs[k].data()); ln.push_back((uint32_t)ref_seqs[k].size()); }
        FILE *fm = fopen(o.meth_out.c_str(), "wb");
        if (!fm) { fprintf(stderr, "failed to open methratio output file: %s\n", o.meth_out.c_str()); return 1; }
        uint64_t st[2] = {0, 0}, nv = 0;
        bsx_meth_valid_count(mh, &nv);
        bsx_meth_write(mh, &o.mo, sp.data(), ln.data(), nullptr, threads, fileno(fm), st);
        fclose(fm);
        printf("total %llu valid mappings, %llu covered cytosines, average coverage: %.2f fold.\n", (unsigned long long)nv, (unsigned long long)st[0],
               st[0] ? (double)st[1] / (double)st[0] : 0.0);
        if (!o.meth_mbias.empty() && bsx_meth_write_mbias_file(mh, o.meth_mbias.c_str()) != BSX_OK) return 1;
        if (o.meth_conv >= 0 && bsx_meth_write_conversion_file(mh, o.meth_conv_report.empty() ? nullptr : o.meth_conv_report.c_str()) != BSX_OK) return 1;
        if (!o.meth_pdr.empty() && bsx_meth_write_pdr_file(mh, &o.mo, sp.data(), ln.data(), nullptr, threads, o.meth_pdr.c_str()) != BSX_OK) return 1;
        if (!o.meth_epialleles.empty() &&
            bsx_meth_write_epialleles_file(mh, &o.mo, sp.data(), ln.data(), nullptr, threads, o.meth_epialleles.c_str()) != BSX_OK) return 1;
        if (!o.meth_mhl.empty() && bsx_meth_write_mhl_file(mh, &o.mo, regions, o.meth_mhl.c_str()) != BSX_OK) return 1;
        if (!o.meth_region_report.empty() && bsx_meth_write_regions_file(mh, &o.mo, regions, o.meth_region_report.c_str()) != BSX_OK) return 1;
        if (timing) fprintf(stderr, "[bsx timing] methratio report %.3f s\n", now() - t);
        bsx_meth_destroy(mh);
    }
    const double tot = (double)(index_a - o.read_start + 1);
    if (pe) printf("Total number of aligned reads: \npairs:       %llu (%.2g%%)\nsingle a:    %llu (%.2g%%)\nsingle b:    %llu (%.2g%%)\n",
                   n_pairs, 100.0 * n_pairs / tot, n_a, 100.0 * n_a / tot, n_b, 100.0 * n_b / tot);
    else printf("Total number of aligned reads: %llu (%.2g%%)\n", n_aligned, 100.0 * n_aligned / tot);
    printf("Done.\n");
    { time_t t = time(nullptr); printf("Finished at %s", ctime(&t)); }
    if (!o.bam_out.empty()) {   // main.cpp:466-473: convert, sort by coordinate, index
        const double t = now();
        printf("Converting SAM to BAM ...\nSorting BAM ...\nIndexing BAM ...\n");
        if (bsx_sam_to_sorted_bam(o.o.c_str(), o.bam_out.c_str(), threads) != BSX_OK) { fprintf(stderr, "%s\n%s remains in SAM format.\n", bsx_last_error(), o.o.c_str()); return 1; }
        remove(o.o.c_str());
        if (timing) fprintf(stderr, "[bsx timing] SAM -> sorted BAM + BAI %.3f s\n", now() - t);
    }
    printf("Total time consumed:  %ld secs\n", (long)(time(nullptr) - t0));
    const double t_fin = now();
    // a stand-alone executable is about to exit: handing 21 GB of device arrays, the pinned slots and the maps back one by one
    // (0.8 s) and then unwinding the CUDA context (1.0 s) buys nothing, the driver reclaims them with the process
    if (!g_exit_after_main) for (int g = n_dev - 1; g >= 0; g--) { bsx_mapper_destroy(mps[g]); bsx_index_destroy(ixs[g]); }
    if (timing) fprintf(stderr, "[bsx timing] teardown %.3f s, total in main %.3f s\n", now() - t_fin, now() - t_start);
    return 0;
}

// called by the executables' main() before bsx_cli_main / bsx_methratio_main: every output is flushed and closed when these
// return, so the process may leave through _exit() without freeing device memory first
extern "C" void bsx_cli_exit_after_main(int on) { g_exit_after_main = on != 0; }
