// bsx_methratio_cli.cpp -- the reference's `methratio.py` command line over the C ABI (SURVEY §8 row f4).
//
//   methratio -o OUT -d REF.fa [-c chr1,chr2] [-u] [-p] [-z] [-q] [-r] [-t N] [-g] [-m FOLD] MAPPING_FILES...
//
// Same options and output as methratio.py:5-16 / 133-154.  Mapping files are BSMAP's SAM (text; FLAG numeric as
// BSMAP writes it, or lettered as `samtools view -X` prints it), BAM (decoded here instead of being piped through
// `samtools view -X`) or BSP output; the format follows the file suffix like the script does.  Text files are
// memory-mapped and parsed on all host threads; the pile-up, and -r's "first alignment in file order wins", run on the
// GPU (bsx_meth.cu).  -s (path to samtools) is accepted and ignored: nothing here shells out.
//
// Extensions (SAM and BAM input only: BSP records carry no read number):
//   --mbias FILE               M-bias report (methylation by read, C context and cycle; include/bsmap_b200.h)
//   --mbias-ignore A,B,C,D     drop calls in the first A / last B cycles of read 1 and first C / last D of read 2
// Extension (SAM, BAM and BSP input):
//   --ct-snp MODE              count C/T SNP evidence from the opposite strand and write the 12-column table with
//                              eff_CT_count, rev_G_count and rev_GA_count; MODE no-action, correct or skip
//   --conversion-filter N      drop alignments with N or more methylated non-CpG calls (incompletely converted reads);
//                              N 0..255, 0 = count only; prints "conversion filter: D of V valid mappings dropped" to stderr
//   --conversion-report FILE   the alignments by their number of methylated non-CpG calls (alone: N = 0)
//   --region-report FILE       methylation levels per region and context (sites, covered, C_count, CT_count, level),
//                              reduced on the device from the same counters as the table, over
//   --regions BED                the regions of a BED file (columns 1-3), in the file's order, or
//   --tiles W                    tiles of W bases over every selected sequence, in the table's order
//   --pdr FILE                 read-level CpG concordance: per CpG position the CpG calls of informative alignments
//                              (at least K CpG calls) that are concordant (all methylated or all unmethylated) or
//                              discordant, and PDR = discordant / (concordant + discordant); prints "PDR: I of V valid
//                              mappings informative (>= K CpG calls), D discordant" to stderr; with --region-report the
//                              report gains the columns concordant, discordant and PDR
//   --pdr-min-cpg K            CpG calls an alignment needs to be informative, 1..255 (default 4)
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <ctime>
#include <string>
#include <unordered_map>
#include <vector>
#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>
#include "bsx_internal.h"

namespace {

struct MOpts {
    std::string out, ref, chroms;
    bsx_meth_opts o;
    bool quiet = false;
    std::string mbias;                       // --mbias FILE
    bool ignore_set = false;
    int32_t ignore[4] = {0, 0, 0, 0};        // --mbias-ignore
    int ct_snp = 0;                          // --ct-snp: BSX_CT_SNP_*
    int conv = -1;                           // --conversion-filter N; -1 = off
    std::string conv_report;                 // --conversion-report FILE
    std::string region_report, regions;      // --region-report FILE, --regions BED
    long long tiles = 0;                     // --tiles W; 0 = none
    std::string pdr;                         // --pdr FILE
    int pdr_min_cpg = 0;                     // --pdr-min-cpg K; 0 = not given (4)
    std::vector<std::string> files;
};

void usage_error(const char *msg) {
    fprintf(stderr, "Usage: methratio [options] BSMAP_MAPPING_FILES\n\nmethratio: error: %s\n", msg);
    exit(2);
}

void disp(const MOpts &m, const char *txt, int nt = 0) {
    if (m.quiet) return;
    time_t t = time(nullptr); char b[64]; strftime(b, sizeof b, "%a %b %e %H:%M:%S %Y", localtime(&t));
    for (int i = 0; i < nt; i++) fputc('\t', stderr);
    fprintf(stderr, "@ %s: %s\n", b, txt);
}

// optparse grammar: -x VAL, -xVAL, --long VAL, --long=VAL; flags may be bundled (-uz)
void parse(int argc, char **argv, MOpts &m) {
    struct Def { char s; const char *l; bool val; };
    static const Def defs[] = {{'o', "out", true}, {'d', "ref", true}, {'c', "chr", true}, {'s', "sam-path", true}, {'u', "unique", false},
                               {'p', "pair", false}, {'z', "zero-meth", false}, {'q', "quiet", false}, {'r', "remove-duplicate", false},
                               {'t', "trim-fillin", true}, {'g', "combine-CpG", false}, {'m', "min-depth", true}, {'h', "help", false},
                               {'\1', "mbias", true}, {'\2', "mbias-ignore", true}, {'\3', "ct-snp", true},
                               {'\4', "conversion-filter", true}, {'\5', "conversion-report", true}, {'\6', "region-report", true},
                               {'\7', "regions", true}, {'\10', "tiles", true}, {'\11', "pdr", true}, {'\12', "pdr-min-cpg", true}};   // long only
    auto apply = [&](char c, const char *v) {
        if (!v) v = "";
        switch (c) {
            case 'o': m.out = v; break;
            case 'd': m.ref = v; break;
            case 'c': m.chroms = v; break;
            case 's': break;                                   // path to samtools: nothing here shells out
            case 'u': m.o.unique = 1; break;
            case 'p': m.o.pair = 1; break;
            case 'z': m.o.meth0 = 1; break;
            case 'q': m.quiet = true; break;
            case 'r': m.o.rm_dup = 1; break;
            case 't': { char *e; long x = strtol(v, &e, 10); if (*e || e == v) usage_error("option -t: invalid integer value"); m.o.trim_fillin = (int)x; } break;
            case 'g': m.o.combine_cpg = 1; break;
            case 'm': { char *e; long x = strtol(v, &e, 10); if (*e || e == v) usage_error("option -m: invalid integer value"); m.o.min_depth = (int)x; } break;
            case '\1': m.mbias = v; break;
            case '\2': {
                const char *q = v;
                for (int k = 0; k < 4; k++) {
                    char *e; const long x = strtol(q, &e, 10);
                    if (e == q || x < 0 || x > 0x7fffffff || *e != (k < 3 ? ',' : '\0')) usage_error("option --mbias-ignore: expected four non-negative integers A,B,C,D");
                    m.ignore[k] = (int32_t)x; q = e + 1;
                }
                m.ignore_set = true;
            } break;
            case '\3':
                m.ct_snp = bsx_ct_snp_mode(v);
                if (!m.ct_snp) usage_error((std::string("option --ct-snp: invalid choice: '") + v + "' (choose from 'no-action', 'correct', 'skip')").c_str());
                break;
            case '\4': { char *e; const long x = strtol(v, &e, 10);
                if (*e || e == v || x < 0 || x > BSX_CONV_BINS - 1) usage_error("option --conversion-filter: expected an integer 0..255");
                m.conv = (int)x; } break;
            case '\5': m.conv_report = v; break;
            case '\6': m.region_report = v; break;
            case '\7': m.regions = v; break;
            case '\10': { char *e; const long long x = strtoll(v, &e, 10);
                if (*e || e == v || x < 1) usage_error("option --tiles: expected an integer >= 1");
                m.tiles = x; } break;
            case '\11': m.pdr = v; break;
            case '\12': { char *e; const long x = strtol(v, &e, 10);
                if (*e || e == v || x < 1 || x > 255) usage_error("option --pdr-min-cpg: expected an integer 1..255");
                m.pdr_min_cpg = (int)x; } break;
            case 'h': printf("Usage: methratio [options] BSMAP_MAPPING_FILES\n  -o FILE -d FILE [-c CHR] [-u] [-p] [-z] [-q] [-r] [-t N] [-g] [-m FOLD] [--mbias FILE] [--mbias-ignore A,B,C,D]\n"
                             "  [--ct-snp no-action|correct|skip] [--conversion-filter N] [--conversion-report FILE]\n"
                             "  [--region-report FILE (--regions BED | --tiles W)] [--pdr FILE [--pdr-min-cpg K]]\n"); exit(0);
        }
    };
    for (int i = 1; i < argc; i++) {
        const char *a = argv[i];
        if (a[0] != '-' || a[1] == 0) { m.files.push_back(a); continue; }
        if (a[1] == '-') {
            if (a[2] == 0) { for (i++; i < argc; i++) m.files.push_back(argv[i]); break; }
            const char *eq = strchr(a, '=');
            const std::string name = eq ? std::string(a + 2, eq) : std::string(a + 2);
            const Def *d = nullptr;
            for (const Def &x : defs) if (name == x.l) d = &x;
            if (!d) usage_error((std::string("no such option: ") + a).c_str());
            if (d->val) { const char *v = eq ? eq + 1 : (i + 1 < argc ? argv[++i] : nullptr); if (!v) usage_error("option requires an argument"); apply(d->s, v); }
            else apply(d->s, nullptr);
            continue;
        }
        for (const char *c = a + 1; *c; c++) {
            const Def *d = nullptr;
            for (const Def &x : defs) if (*c == x.s && *c > ' ') d = &x;
            if (!d) usage_error((std::string("no such option: -") + *c).c_str());
            if (d->val) { const char *v = c[1] ? c + 1 : (i + 1 < argc ? argv[++i] : nullptr); if (!v) usage_error("option requires an argument"); apply(d->s, v); break; }
            apply(d->s, nullptr);
        }
    }
}

struct Aln { const char *seq; uint32_t len, chr, pos; int32_t insert, mate; uint8_t strand, flags; };

struct Field { const char *p; uint32_t n; };
// split [b, e) at tabs into at most cap fields; returns the count
inline int split(const char *b, const char *e, Field *f, int cap) {
    int n = 0;
    const char *s = b;
    while (n < cap) {
        const char *t = (const char *)memchr(s, '\t', (size_t)(e - s));
        if (!t) { f[n++] = Field{s, (uint32_t)(e - s)}; break; }
        f[n++] = Field{s, (uint32_t)(t - s)};
        s = t + 1;
    }
    return n;
}
inline long long to_int(Field f) { long long v = 0; bool neg = false; uint32_t i = 0; if (i < f.n && (f.p[i] == '-' || f.p[i] == '+')) { neg = f.p[i] == '-'; i++; } for (; i < f.n && f.p[i] >= '0' && f.p[i] <= '9'; i++) v = v * 10 + (f.p[i] - '0'); return neg ? -v : v; }

// get_alignment (methratio.py:30-54) up to the point where the device takes over
bool parse_line(const char *b, const char *e, bool sam, const std::unordered_map<std::string, uint32_t> &chrom, Aln &a, std::string &err) {
    if (e > b && e[-1] == '\r') e--;
    Field f[64];
    if (sam) {
        if (b < e && *b == '@') return false;
        const int n = split(b, e, f, 64);
        if (n < 11) return false;
        uint32_t fl = 0;
        // numeric when every character is a digit: the letters of 0x40 / 0x80 ('1', '2') may open a lettered FLAG ("2s")
        bool numeric = f[1].n > 0;
        for (uint32_t i = 0; i < f[1].n; i++) numeric = numeric && f[1].p[i] >= '0' && f[1].p[i] <= '9';
        if (numeric) {
            const long long v = to_int(f[1]);
            if (v & 0x4) return false;
            if (v & 0x100) fl |= BSX_METH_SECONDARY;
            if (v & 0x2) fl |= BSX_METH_PROPER;
            if (v & 0x80) fl |= BSX_METH_READ2;
        } else {
            for (uint32_t i = 0; i < f[1].n; i++) {
                const char c = f[1].p[i];
                if (c == 'u') return false;
                if (c == 's') fl |= BSX_METH_SECONDARY;
                if (c == 'P') fl |= BSX_METH_PROPER;
                if (c == '2') fl |= BSX_METH_READ2;
            }
        }
        auto it = chrom.find(std::string(f[2].p, f[2].n));
        if (it == chrom.end()) return false;
        int strand = -1;
        for (int k = 11; k < n; k++)
            if (f[k].n >= 7 && memcmp(f[k].p, "ZS:Z:", 5) == 0) { strand = (f[k].p[5] == '-' ? 1 : 0) | (f[k].p[6] == '-' ? 2 : 0); break; }
        if (strand < 0) { err = "SAM line without a ZS:Z: tag (not BSMAP output?)"; return false; }
        a.seq = f[9].p; a.len = f[9].n; a.chr = it->second; a.pos = (uint32_t)(to_int(f[3]) - 1);
        a.insert = (int32_t)to_int(f[8]); a.mate = (int32_t)(to_int(f[7]) - 1);
        a.strand = (uint8_t)strand; a.flags = (uint8_t)(fl | BSX_METH_SAM);
        return true;
    }
    const int n = split(b, e, f, 64);
    if (n < 4 || f[3].n < 2) return false;
    if ((f[3].p[0] == 'N' && f[3].p[1] == 'M') || (f[3].p[0] == 'Q' && f[3].p[1] == 'C')) return false;
    if (n < 8) return false;
    uint32_t fl = 0;
    if (!(f[3].p[0] == 'U' && f[3].p[1] == 'M')) fl |= BSX_METH_SECONDARY;
    if (!(f[7].n == 1 && f[7].p[0] == '0')) fl |= BSX_METH_PROPER;
    auto it = chrom.find(std::string(f[4].p, f[4].n));
    if (it == chrom.end()) return false;
    a.seq = f[1].p; a.len = f[1].n; a.chr = it->second; a.pos = (uint32_t)(to_int(f[5]) - 1);
    a.insert = (int32_t)to_int(f[7]); a.mate = 0;
    a.strand = (uint8_t)((f[6].n > 0 && f[6].p[0] == '-' ? 1 : 0) | (f[6].n > 1 && f[6].p[1] == '-' ? 2 : 0)); a.flags = (uint8_t)fl;
    return true;
}

// A BAM file (the script reads it through `samtools view -X`, methratio.py:91): reference names from the file's own
// dictionary, FLAG bits 0x4 / 0x100 / 0x2 = the letters u / s / P, SEQ through the 4-bit table, ZS:Z from the tags.
// Records are found with one sequential hop over the block sizes, then decoded in parallel, PIECE records at a time.
template <class Pile>
bool pile_bam(const std::string &path, const std::unordered_map<std::string, uint32_t> &chrom, int threads, Pile &pile, std::string &err) {
    std::vector<char> raw;
    if (bsx_inflate_file(path.c_str(), raw) != BSX_OK) { err = "failed to read (BGZF inflate)"; return false; }
    const unsigned char *p = (const unsigned char *)raw.data();
    const size_t n = raw.size();
    auto i32 = [&](size_t at) { int32_t v; memcpy(&v, p + at, 4); return v; };
    if (n < 12 || memcmp(p, "BAM\1", 4) != 0) { err = "not a BAM file"; return false; }
    size_t at = 8 + (size_t)std::max(i32(4), 0);
    if (at + 4 > n) { err = "truncated BAM header"; return false; }
    const int32_t n_ref = i32(at); at += 4;
    std::vector<int64_t> ref_to_chr((size_t)std::max(n_ref, 0), -1);       // BAM refID -> index of the FASTA record (or not selected)
    for (int32_t k = 0; k < n_ref; k++) {
        if (at + 4 > n) { err = "truncated BAM header"; return false; }
        const int32_t l_name = i32(at);
        if (l_name < 1 || at + 4 + (size_t)l_name + 4 > n) { err = "truncated BAM header"; return false; }
        auto it = chrom.find(std::string((const char *)p + at + 4, (size_t)l_name - 1));
        if (it != chrom.end()) ref_to_chr[(size_t)k] = it->second;
        at += 4 + (size_t)l_name + 4;
    }
    static const char nt16[] = "=ACMGRSVTWYHKDBN";
    const size_t PIECE = (size_t)4 << 20;
    while (at + 4 <= n) {
        std::vector<size_t> recs;                                            // offsets of the records' bodies
        while (recs.size() < PIECE && at + 4 <= n) {
            const int32_t bs = i32(at);
            if (bs < 32 || at + 4 + (size_t)bs > n) { err = "truncated BAM record"; return false; }
            recs.push_back(at + 4); at += 4 + (size_t)bs;
        }
        std::vector<std::vector<Aln>> part((size_t)threads);
        std::vector<std::vector<char>> bases((size_t)threads);
        std::vector<std::string> errs((size_t)threads);
        bsx_parallel(threads, recs.size(), [&](int t, size_t b, size_t e) {
            size_t need = 0;
            for (size_t r = b; r < e; r++) need += (size_t)std::max(i32(recs[r] + 16), 0);
            bases[t].resize(need + 1);                                       // decoded SEQ of this thread's records, never reallocated
            size_t used = 0;
            for (size_t r = b; r < e; r++) {
                const unsigned char *q = p + recs[r];
                const size_t bytes = (size_t)i32(recs[r] - 4);
                const int32_t ref_id = i32(recs[r]), pos = i32(recs[r] + 4), l_seq = i32(recs[r] + 16), next_pos = i32(recs[r] + 24), tlen = i32(recs[r] + 28);
                const uint32_t l_name = q[8], n_cig = (uint32_t)q[12] | ((uint32_t)q[13] << 8), flag = (uint32_t)q[14] | ((uint32_t)q[15] << 8);
                const size_t off_seq = 32 + (size_t)l_name + 4 * (size_t)n_cig;
                if (l_seq < 0 || off_seq + ((size_t)l_seq + 1) / 2 + (size_t)l_seq > bytes) { errs[t] = "truncated BAM record"; return; }
                if (flag & 0x4) continue;                                    // 'u'
                if (ref_id < 0 || ref_id >= (int32_t)ref_to_chr.size() || ref_to_chr[(size_t)ref_id] < 0) continue;   // cr not in options.chroms
                Aln a;
                a.flags = (uint8_t)(BSX_METH_SAM | ((flag & 0x100) ? BSX_METH_SECONDARY : 0u) | ((flag & 0x2) ? BSX_METH_PROPER : 0u) |
                                   ((flag & 0x80) ? BSX_METH_READ2 : 0u));
                a.chr = (uint32_t)ref_to_chr[(size_t)ref_id]; a.pos = (uint32_t)pos; a.insert = tlen; a.mate = next_pos;
                char *sq = bases[t].data() + used;
                for (int32_t i = 0; i < l_seq; i++) sq[i] = nt16[(q[off_seq + ((size_t)i >> 1)] >> ((~i & 1) << 2)) & 15];
                a.seq = sq; a.len = (uint32_t)l_seq; used += (size_t)l_seq;
                if (l_seq == 0) { a.seq = "*"; a.len = 1; }                 // no SEQ: `samtools view` prints '*', one character to the script
                // tags: two letters, a type, a value
                int strand = -1;
                size_t x = off_seq + ((size_t)l_seq + 1) / 2 + (size_t)l_seq;
                while (x + 3 <= bytes && strand < 0) {
                    const char t0 = (char)q[x], t1 = (char)q[x + 1], ty = (char)q[x + 2];
                    x += 3;
                    if (ty == 'Z' || ty == 'H') {
                        const void *z = memchr(q + x, 0, bytes - x);
                        const size_t l = z ? (size_t)((const unsigned char *)z - (q + x)) : bytes - x;
                        if (t0 == 'Z' && t1 == 'S' && ty == 'Z' && l >= 2) strand = (q[x] == '-' ? 1 : 0) | (q[x + 1] == '-' ? 2 : 0);
                        x += l + 1;
                    } else if (ty == 'A' || ty == 'c' || ty == 'C') x += 1;
                    else if (ty == 's' || ty == 'S') x += 2;
                    else if (ty == 'i' || ty == 'I' || ty == 'f') x += 4;
                    else if (ty == 'B' && x + 5 <= bytes) {
                        const char sub = (char)q[x]; uint32_t cnt; memcpy(&cnt, q + x + 1, 4);
                        x += 5 + (size_t)cnt * (sub == 'c' || sub == 'C' ? 1u : (sub == 's' || sub == 'S' ? 2u : 4u));
                    } else break;
                }
                if (strand < 0) { errs[t] = "BAM record without a ZS:Z: tag (not BSMAP output?)"; return; }
                a.strand = (uint8_t)strand;
                part[t].push_back(a);
            }
        });
        for (const std::string &e : errs) if (!e.empty()) { err = e; return false; }
        if (!pile(part)) return false;
    }
    return true;
}

}  // namespace

static double now_s() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

extern "C" int bsx_methratio_main(int argc, char **argv) {
    const double t_start = now_s();
    MOpts m; bsx_meth_opts_default(&m.o);
    parse(argc, argv, m);
    if (m.ref.empty()) usage_error("Missing reference file, use -d or --ref option.");
    if (m.out.empty()) usage_error("Missing output file name, use -o or --out option.");
    if (m.files.empty()) usage_error("Require at least one BSMAP_MAPPING_FILE.");
    if (!m.conv_report.empty() && m.conv < 0) m.conv = 0;
    if (!m.regions.empty() && m.tiles) usage_error("--regions and --tiles exclude each other");
    if (m.region_report.empty() && (!m.regions.empty() || m.tiles)) usage_error("--regions / --tiles need --region-report FILE");
    if (!m.region_report.empty() && m.regions.empty() && !m.tiles) usage_error("--region-report needs --regions BED or --tiles W");
    if (m.pdr_min_cpg && m.pdr.empty()) usage_error("--pdr-min-cpg needs --pdr FILE");
    if (!m.pdr.empty() && !m.pdr_min_cpg) m.pdr_min_cpg = 4;
    const bool cycles = !m.mbias.empty() || m.ignore_set;
    if (cycles)
        for (const std::string &f : m.files) {
            std::string suf = f.size() >= 4 ? f.substr(f.size() - 4) : "";
            for (char &c : suf) c = (char)toupper((unsigned char)c);
            if (suf != ".SAM" && suf != ".BAM") usage_error(("--mbias / --mbias-ignore need SAM or BAM input (BSP records carry no read number): " + f).c_str());
        }
    const int threads = bsx_host_threads(0);

    disp(m, ("reading reference " + m.ref + " ...").c_str());
    std::thread ctx_thread([] { cudaFree(nullptr); });        // the CUDA context comes up while the FASTA is parsed
    std::vector<std::string> names, seqs;
    const int lrc = bsx_load_fasta(m.ref.c_str(), names, seqs);
    const double t_fa = now_s();
    ctx_thread.join();
    const double t_ctx = now_s();
    if (lrc != BSX_OK) { fprintf(stderr, "%s\n", bsx_last_error()); return 1; }
    // -c: only these chromosomes (methratio.py:74-79); mappings to any other name are skipped
    std::vector<uint8_t> selected(names.size(), 1);
    if (!m.chroms.empty()) {
        std::fill(selected.begin(), selected.end(), 0);
        size_t s = 0;
        while (s <= m.chroms.size()) {
            size_t e = m.chroms.find(',', s); if (e == std::string::npos) e = m.chroms.size();
            const std::string want = m.chroms.substr(s, e - s);
            for (size_t k = 0; k < names.size(); k++) if (names[k] == want) selected[k] = 1;
            s = e + 1;
        }
    }
    std::unordered_map<std::string, uint32_t> chrom;
    for (size_t k = 0; k < names.size(); k++) if (selected[k]) chrom[names[k]] = (uint32_t)k;   // a repeated name: the last record wins, as in the dict

    std::vector<const char *> np, sp; std::vector<uint32_t> ln;
    for (size_t k = 0; k < seqs.size(); k++) { np.push_back(names[k].c_str()); sp.push_back(seqs[k].data()); ln.push_back((uint32_t)seqs[k].size()); }
    bsx_index *ix = nullptr; bsx_meth *mh = nullptr;
    if (bsx_index_create_packed((int)seqs.size(), np.data(), sp.data(), ln.data(), 0, &ix) != BSX_OK || bsx_meth_create(ix, &mh) != BSX_OK) {
        fprintf(stderr, "%s\n", bsx_last_error()); return 1; }
    if ((!m.mbias.empty() && bsx_meth_enable_mbias(mh) != BSX_OK) || (m.ignore_set && bsx_meth_set_ignore(mh, m.ignore) != BSX_OK) ||
        (m.ct_snp && bsx_meth_enable_ct_snp(mh, m.ct_snp) != BSX_OK) || (m.conv >= 0 && bsx_meth_enable_conversion_filter(mh, m.conv) != BSX_OK) ||
        (!m.pdr.empty() && bsx_meth_enable_pdr(mh, m.pdr_min_cpg) != BSX_OK)) {
        fprintf(stderr, "%s\n", bsx_last_error()); return 1; }
    bsx_regions regions;                                      // read before the pile-up, so that a bad BED fails early
    if ((!m.regions.empty() && bsx_regions_bed(ix, selected.data(), m.regions.c_str(), regions) != BSX_OK) ||
        (m.tiles && bsx_regions_tiles(ix, selected.data(), (uint64_t)m.tiles, regions) != BSX_OK)) {
        fprintf(stderr, "%s\n", bsx_last_error()); return 1; }

    const double t_ix = now_s();
    uint64_t nmap = 0;
    const char *cur_path = "";
    // one piece of alignments (file order = thread 0's, then thread 1's, ...) -> staging arrays -> the device
    auto pile = [&](const std::vector<std::vector<Aln>> &part) -> bool {
        size_t tot = 0; uint32_t maxlen = 16;
        std::vector<size_t> off((size_t)threads + 1, 0);
        for (int t = 0; t < threads; t++) { off[t] = tot; tot += part[t].size(); for (const Aln &a : part[t]) maxlen = std::max(maxlen, a.len); }
        off[threads] = tot;
        if (tot > 0xffffffffull) { fprintf(stderr, "too many alignments in one piece\n"); return false; }
        // bsx_meth_add takes 16-bit lengths: a longer SEQ is refused rather than piled up cut short
        if (maxlen > 65535u) { fprintf(stderr, "%s: SEQ longer than 65535 bases (%u): not supported\n", cur_path, maxlen); return false; }
        const uint32_t stride = (maxlen + 15u) & ~15u;
        std::vector<char> sq(tot * stride); std::vector<uint16_t> len(tot); std::vector<uint32_t> chr(tot), pos(tot);
        std::vector<uint8_t> strand(tot), flags(tot); std::vector<int32_t> ins(tot), mate(tot);
        bsx_parallel(threads, (size_t)threads, [&](int t, size_t, size_t) {
            size_t i = off[t];
            for (const Aln &a : part[t]) {
                memcpy(&sq[i * stride], a.seq, a.len);
                len[i] = (uint16_t)a.len; chr[i] = a.chr; pos[i] = a.pos; strand[i] = a.strand; flags[i] = a.flags; ins[i] = a.insert; mate[i] = a.mate;
                i++;
            }
        });
        if (bsx_meth_add(mh, &m.o, (uint32_t)tot, sq.data(), stride, len.data(), chr.data(), pos.data(), strand.data(), ins.data(), mate.data(),
                         flags.data(), &nmap) != BSX_OK) { fprintf(stderr, "%s\n", bsx_last_error()); return false; }
        return true;
    };
    for (const std::string &path : m.files) {
        disp(m, ("reading " + path + " ...").c_str());
        cur_path = path.c_str();
        const size_t pl = path.size();
        std::string suf = pl >= 4 ? path.substr(pl - 4) : "";
        for (char &c : suf) c = (char)toupper((unsigned char)c);
        if (suf == ".BAM") {
            // methratio.py:91 pipes the file through `samtools view -X`; here the records are decoded in place
            std::string err;
            if (!pile_bam(path, chrom, threads, pile, err)) { if (!err.empty()) fprintf(stderr, "%s: %s\n", path.c_str(), err.c_str()); return 1; }
            continue;
        }
        const bool sam = suf == ".SAM";
        const int fd = open(path.c_str(), O_RDONLY);
        struct stat st;
        if (fd < 0 || fstat(fd, &st) != 0) { fprintf(stderr, "failed to open mapping file: %s\n", path.c_str()); return 1; }
        const size_t n = (size_t)st.st_size;
        if (n == 0) { close(fd); continue; }
        const char *p = (const char *)mmap(nullptr, n, PROT_READ, MAP_PRIVATE, fd, 0);
        if (p == MAP_FAILED) { fprintf(stderr, "mmap failed: %s\n", path.c_str()); return 1; }
        madvise((void *)p, n, MADV_SEQUENTIAL);
        // byte ranges cut at line starts, one per thread and ~64 MB piece; parsed in parallel, piled up piece by piece
        const size_t PIECE = (size_t)256 << 20;
        for (size_t p0 = 0; p0 < n;) {
            size_t p1 = std::min(n, p0 + PIECE);
            if (p1 < n) { const void *q = memchr(p + p1, '\n', n - p1); p1 = q ? (size_t)((const char *)q - p) + 1 : n; }
            const int threads_here = (p1 - p0) < ((size_t)1 << 20) ? 1 : threads;   // tiny pieces: one thread, no boundary games
            std::vector<std::vector<Aln>> part((size_t)threads);
            std::vector<std::string> errs((size_t)threads);
            bsx_parallel(threads_here, (size_t)threads_here, [&, threads_here](int t, size_t, size_t) {
                const int threads = threads_here;
                size_t b = p0 + (p1 - p0) * (size_t)t / threads, e = p0 + (p1 - p0) * (size_t)(t + 1) / threads;
                if (t > 0) { const void *q = memchr(p + b - 1, '\n', p1 - (b - 1)); b = q ? (size_t)((const char *)q - p) + 1 : p1; }   // first line start at or after b
                if (t + 1 < threads && e > p0) { const void *q = memchr(p + e - 1, '\n', p1 - (e - 1)); e = q ? (size_t)((const char *)q - p) + 1 : p1; }
                part[t].reserve((e > b ? e - b : 0) / 200 + 16);
                while (b < e) {
                    const void *q = memchr(p + b, '\n', p1 - b);
                    const size_t le = q ? (size_t)((const char *)q - p) : p1;
                    Aln a;
                    if (le > b && parse_line(p + b, p + le, sam, chrom, a, errs[t])) part[t].push_back(a);
                    b = le + 1;
                }
            });
            for (const std::string &e : errs) if (!e.empty()) { fprintf(stderr, "%s: %s\n", path.c_str(), e.c_str()); return 1; }
            if (!pile(part)) return 1;
            p0 = p1;
        }
        munmap((void *)p, n); close(fd);
    }
    const double t_pile = now_s();
    if (m.o.combine_cpg) disp(m, "combining CpG methylation from both strands ...");
    disp(m, ("writing " + m.out + " ...").c_str());
    const int ofd = open(m.out.c_str(), O_WRONLY | O_CREAT | O_TRUNC, 0644);
    if (ofd < 0) { fprintf(stderr, "failed to open output file: %s\n", m.out.c_str()); return 1; }
    uint64_t stats[2] = {0, 0};
    bsx_meth_write(mh, &m.o, sp.data(), ln.data(), selected.data(), threads, ofd, stats);
    close(ofd);
    if (!m.mbias.empty()) {
        disp(m, ("writing " + m.mbias + " ...").c_str());
        if (bsx_meth_write_mbias_file(mh, m.mbias.c_str()) != BSX_OK) return 1;
    }
    if (m.conv >= 0) {
        if (!m.conv_report.empty()) disp(m, ("writing " + m.conv_report + " ...").c_str());
        if (bsx_meth_write_conversion_file(mh, m.conv_report.empty() ? nullptr : m.conv_report.c_str()) != BSX_OK) return 1;
    }
    if (!m.pdr.empty()) {
        disp(m, ("writing " + m.pdr + " ...").c_str());
        if (bsx_meth_write_pdr_file(mh, &m.o, sp.data(), ln.data(), selected.data(), threads, m.pdr.c_str()) != BSX_OK) return 1;
    }
    if (!m.region_report.empty()) {
        disp(m, ("writing " + m.region_report + " ...").c_str());
        if (bsx_meth_write_regions_file(mh, &m.o, regions, m.region_report.c_str()) != BSX_OK) return 1;
    }
    if (getenv("BSX_CLI_TIMING"))
        fprintf(stderr, "[bsx timing] reference FASTA %.3f s || CUDA context (ready at %.3f s), packed reference + counters %.3f s, parse + pile-up %.3f s, report %.3f s\n",
                t_fa - t_start, t_ctx - t_start, t_ix - t_ctx, t_pile - t_ix, now_s() - t_pile);
    disp(m, "done.");
    printf("total %llu valid mappings, %llu covered cytosines, average coverage: %.2f fold.\n", (unsigned long long)nmap,
           (unsigned long long)stats[0], stats[0] ? (double)stats[1] / (double)stats[0] : 0.0);
    bsx_meth_destroy(mh); bsx_index_destroy(ix);
    return 0;
}
