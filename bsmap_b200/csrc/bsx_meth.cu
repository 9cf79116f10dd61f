// bsx_meth.cu -- methratio.py on the device (SURVEY §8 row f4): per-position methylation counters piled up from
// the mappings by a warp-per-alignment kernel with global atomics, CpG combining, and the host report writer.
//
// Reference: methratio.py.  get_alignment (30-65): filters, fill-in trimming, mate-overlap removal;
// pile-up (95-118): on a '+' (Watson) hit every reference C under the read counts T as depth and C as
// meth + depth, on a '-' (Crick) hit every reference G counts A / G; -g (122-131); report (133-154).
// The reference holds two u32 arrays per chromosome in host memory and walks each read with str.find;
// here both arrays cover the packed Watson strand of the index in HBM (8 bytes per reference position) and the
// reference base comes from the 2-bit refcat (non-ACGT packs to A, which is neither C nor G -- same outcome).
// -r (methratio.py:52-55: of the alignments that pass the filters, the first in file order per (chromosome, fragment
// end, direction) counts) is a two-kernel min-reduction: every alignment of a batch claims its key with
// atomicMin(first[key], order + 1), then the pile-up kernel lets the alignment through whose claim stands and marks
// the key 0 = taken for good, so later batches lose against earlier ones.  8 bytes per reference position, allocated
// on first use.
//
// M-bias (bsx_meth_enable_mbias) and per-cycle exclusion (bsx_meth_set_ignore) switch both pile-up kernels to their
// `Cycles` instantiation: each call also gets its cycle (position in the read as sequenced), read (1 / 2) and C context
// (CpG / CHG / CHH), excluded calls are dropped from the counters, and the others go into a per-CTA shared-memory
// histogram [read][context][cycle][meth|unmeth] that is flushed (non-zero bins only) into a device-global u64 one.  That
// grid is capped at the resident CTAs and strides over the alignments, so one flush serves many alignments.  With both
// off the kernels are the plain instantiation, which compiles to the same code as before these options existed.
//
// C/T SNP evidence (bsx_meth_enable_ct_snp) switches them to their `Snp` instantiation: a base under the read whose
// reference code is the complement of the call's (G under a '+' hit, C under a '-' hit) is opposite-strand evidence,
// untouched by bisulfite: the read shows G / C when the genome has the reference C, A / T when it has a T (a C/T SNP).
// Two more u32 arrays over the same positions count those bases, `confirm` and `snp`, one global atomic per counted
// base.  The writer then scales or drops a C's line by that evidence.
//
// The conversion filter (bsx_meth_enable_conversion_filter) switches them to their `Conv` instantiation, which exists only
// with `Cycles` (it needs the call's cycle and context, and its histogram the capped grid): before an alignment's calls are
// deposited, the warp counts its methylated non-CpG calls (its score), lane 0 adds the alignment to a per-CTA shared
// histogram of scores, and an alignment whose score reaches the threshold returns without depositing anything.
//
// The proportion of discordant reads (bsx_meth_enable_pdr) switches them to their `Pdr` instantiation, again only with
// `Cycles`: the same first pass also counts the alignment's methylated and unmethylated CpG calls, and when there are at
// least K of them the second pass adds every CpG call to `concordant` (all methylated or all unmethylated) or
// `discordant`, two more u32 arrays over the positions.  The informative and discordant alignments go into two per-CTA
// shared counters, flushed like the histograms.
//
// 4-CpG epialleles (bsx_meth_enable_epialleles) switch them to their `Epi` instantiation, again only with `Cycles`.  A
// CpG rank index over the packed reference (one u32 per word: the CpG sites before it; built on the device by a counting
// kernel and a scan) numbers the sites, and 16 u32 counters per site count the methylation patterns of the alignments
// that carry a call at that site and the next three.  The first pass counts the alignment's CpG calls; one with at least
// four walks its span again, 32 positions a step, with three ballots (site, call, methylated) and the last three sites'
// bits carried from step to step in warp-uniform registers.  The lane whose call closes a fully called run of four adds
// the pattern to the first site's row: one global atomic per window.
//
// Methylation haplotype load (bsx_meth_enable_mhl) rides on the same walk (the Epi instantiation, with EpiArgs::mhl
// set; an alignment with one CpG call is walked): 48 u32 counters per site count, by run length capped at 16, the
// alignments in which a run of called / methylated / unmethylated sites ends there.  A called lane's runs are the sites
// since the step's last break below it, plus the warp-uniform carries when there is none; it adds to family 0 and to 1
// or 2: two global atomics per call.  meth_mhl_region_kernel reduces them over regions: each region's rank range from
// the index, chunks of MHL_CHUNK ranks per warp, lanes over (site, run length), and a suffix sum over the run lengths.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <string>
#include <unordered_map>
#include <vector>
#include <fcntl.h>
#include <unistd.h>
#include "bsx_internal.h"
#include "bsx_common.cuh"

struct bsx_meth {
    const bsx_index *ix = nullptr;
    uint32_t *d_meth = nullptr, *d_depth = nullptr;   // n_words * 16 counters each, indexed like refcat bases
    unsigned long long *d_valid = nullptr;
    uint32_t *d_first = nullptr;                      // -r: per (position, direction) the order + 1 of the claiming alignment; 0 = taken
    cudaEvent_t dup_order = nullptr;                  // -r, in-process: the pile-up of batch k+1 waits for that of batch k
    bool combined = false;
    // staging for bsx_meth_add
    size_t cap = 0; uint32_t stride = 0;
    char *d_seq = nullptr; uint16_t *d_len = nullptr; uint32_t *d_chr = nullptr, *d_pos = nullptr;
    uint8_t *d_strand = nullptr, *d_flags = nullptr; int32_t *d_ins = nullptr, *d_mate = nullptr;
    // M-bias / exclusion: fixed before the first alignment is piled up
    bool mbias = false, started = false;
    int32_t ignore[4] = {0, 0, 0, 0};                 // r1_5p, r1_3p, r2_5p, r2_3p
    unsigned long long *d_mbias = nullptr;            // MBIAS_BINS counters, then the overflow counter
    int resident[2] = {0, 0};                         // CTAs of the Cycles pile-up kernels (text, mapped) the device holds at once
    // C/T SNP evidence: fixed before the first alignment is piled up
    int ct_snp = 0;                                   // BSX_CT_SNP_*, 0 = off
    uint32_t *d_confirm = nullptr, *d_snp = nullptr;  // n_words * 16 counters each, like d_meth / d_depth
    // conversion filter: fixed before the first alignment is piled up
    int conv_threshold = 0;                           // 0 = report only
    unsigned long long *d_conv = nullptr;             // BSX_CONV_BINS alignments by score; NULL = filter off
    // PDR: fixed before the first alignment is piled up
    uint32_t pdr_min_cpg = 0;                         // K; 0 = off
    uint32_t *d_conc = nullptr, *d_disc = nullptr;    // n_words * 16 counters each, like d_meth / d_depth
    unsigned long long *d_pdr = nullptr;              // informative, discordant alignments; NULL = PDR off
    // epialleles: fixed before the first alignment is piled up
    uint32_t *d_cpg_rank = nullptr;                   // n_words + 1: the CpG sites before each word (the last: all of them)
    uint32_t *d_epi = nullptr;                        // 16 counters per site, by pattern; NULL = epialleles off
    unsigned long long *d_epi_count = nullptr;        // alignments with a window, windows counted
    uint64_t cpg_sites = 0;
    // MHL: fixed before the first alignment is piled up
    uint32_t *d_mhl = nullptr;                        // 48 counters per site, [family][run length - 1]; NULL = MHL off
    unsigned long long *d_mhl_count = nullptr;        // alignments with a CpG call, CpG calls
};

namespace {

constexpr int MBIAS_BINS = 2 * 3 * BSX_MBIAS_CYCLES * 2;

// what the Cycles instantiation needs beyond the plain one
struct MbiasArgs {
    unsigned long long *hist;     // MBIAS_BINS counters, then the overflow counter (calls at cycle >= BSX_MBIAS_CYCLES);
                                  // NULL: exclusion only, no histogram to keep
    int32_t ignore[4];            // r1_5p, r1_3p, r2_5p, r2_3p
    int readset;                  // mapped single-end batches: 2 = these are read 2
};

// what the Conv instantiation needs beyond the Cycles one
struct ConvArgs {
    unsigned long long *hist;     // BSX_CONV_BINS valid alignments by score (the last bin: BSX_CONV_BINS - 1 or more)
    uint32_t threshold;           // an alignment with score >= threshold is dropped; 0 = none is
};

// what the Pdr instantiation needs beyond the Cycles one
struct PdrArgs {
    uint32_t *concordant, *discordant;   // per position: CpG calls of informative alignments, by the alignment's class
    unsigned long long *count;           // informative, discordant alignments
    uint32_t min_cpg;                    // K: an alignment with K or more CpG calls is informative
};

// what the Epi instantiation needs beyond the Cycles one
struct EpiArgs {
    const uint32_t *rank;                // per packed word: the CpG sites before it
    uint32_t *counts;                    // 16 per site: the windows starting there, by pattern; NULL = MHL only
    unsigned long long *count;           // alignments with a window, windows counted
    uint32_t *mhl;                       // 48 per site: runs ending there, [family][length - 1]; NULL = MHL off
    unsigned long long *mhl_count;       // alignments with a CpG call, CpG calls
};

// Conv: the CTA's alignments by score, zeroed before and flushed (non-zero bins) after them.  At file scope, so that the
// pile-up addresses it directly; only the Conv kernels reference it, and only they are given its 1 KB.
__shared__ uint32_t conv_hist[BSX_CONV_BINS];
// Pdr: the CTA's informative and discordant alignments, zeroed and flushed the same way
__shared__ uint32_t pdr_count[2];
// Epi: the CTA's alignments with a window and its windows, zeroed and flushed the same way
__shared__ uint32_t epi_count[2];
// MHL (Epi with EpiArgs::mhl): the CTA's alignments with a CpG call and their calls, zeroed and flushed the same way
__shared__ uint32_t mhl_count[2];

__device__ __forceinline__ uint32_t ref_code(const uint32_t *refcat, uint32_t q) { return (refcat[q >> 4] >> (30 - 2 * (q & 15))) & 3u; }

// the CpG sites of a packed word w: bit 30 - 2j set when base j is C and base j + 1 is G (for j = 15, the first base of
// the next word nx)
__host__ __device__ __forceinline__ uint32_t cpg_mask(uint32_t w, uint32_t nx) {
    const uint32_t lo = w & 0x55555555u, hi = (w >> 1) & 0x55555555u;
    return (lo & ~hi) & (((hi & ~lo) << 2) | ((nx >> 30) == 2u ? 1u : 0u));
}
// the rank of CpG site c (its C's position): the sites before its word, then those before it in the word (they end
// inside the word, so the next word is not needed)
__device__ __forceinline__ uint32_t cpg_rank(const uint32_t *__restrict__ refcat, const uint32_t *__restrict__ rank, uint32_t c) {
    return __ldg(rank + (c >> 4)) + __popc(cpg_mask(__ldg(refcat + (c >> 4)), 0u) & ~(0xffffffffu >> (2 * (c & 15))));
}

// Epi's third pass over an alignment's trimmed span [0, len) (read offset start + i, printed length L; calls of cycles
// outside [lo, hi) are excluded), 32 positions a step with every lane active.  A site of the alignment's strand is a
// '+' C whose next base is G (the site is the C) or a '-' G whose previous base is C (the site is that C); its call is
// the read's methylated or converted letter in the cycle bounds, anything else breaks the windows through the site.
// Three ballots mark the step's sites, calls and methylated calls; c3 / m3 carry the called / methylated bits of the last
// three sites before the step (bit t: the (t + 1)-th latest), warp-uniform.  A called lane whose three previous sites are
// called closes a window: its pattern is the four methylated bits, the earliest site the most significant, and its row
// the earliest site's rank, so rank - 3.  Lane 0 counts the alignment and its windows in epi_count (shared).
// MHL (ep.mhl): run[f] carries the length (capped at 16) of the run of family f (called, methylated, unmethylated) that
// ends at the last site before the step; a called lane's run is the sites after the latest break below it in the step,
// plus run[f] when there is none, plus itself.  ep.counts NULL: no windows.
template <class GetC>
__device__ __forceinline__ void epi_windows(const uint32_t *__restrict__ refcat, uint32_t base, int len, int start, int L, bool rev, int lo, int hi,
                                            bool first_minus, uint32_t match, char cm, char cc, int lane, GetC getc, const EpiArgs &ep) {
    const uint32_t want = 3u - match, below = (1u << lane) - 1u;
    uint32_t c3 = 0u, m3 = 0u, mine = 0u, run[3] = {0u, 0u, 0u}, ncalls = 0u;
    // the called / methylated bits of the three latest sites among `sites`, then those carried in
    auto last3 = [&](uint32_t sites, uint32_t calls, uint32_t meths, uint32_t &c, uint32_t &mm) {
        uint32_t cn = 0u, mn = 0u, t = 0u;
#pragma unroll
        for (int r = 0; r < 3; r++) {
            if (!sites) break;
            const int p = 31 - __clz(sites);
            sites &= ~(1u << p);
            cn |= ((calls >> p) & 1u) << t; mn |= ((meths >> p) & 1u) << t; t++;
        }
        c = (cn | (c3 << t)) & 7u; mm = (mn | (m3 << t)) & 7u;
    };
#pragma unroll 1
    for (int i0 = 0; i0 < len; i0 += 32) {
        const int i = i0 + lane;
        const uint32_t q = base + (uint32_t)i;
        bool site = false, called = false, is_m = false;
        if (i < len && ref_code(refcat, q) == match) {
            site = (first_minus ? ref_code(refcat, q - 1u) : ref_code(refcat, q + 1u)) == want;
            if (site) {
                const int j = start + i;
                const char c = getc(j);
                const int cyc = rev ? L - 1 - j : j;
                called = (c == cm || c == cc) && cyc >= lo && cyc < hi;
                is_m = called && c == cm;
            }
        }
        const uint32_t sites = __ballot_sync(0xffffffffu, site), calls = __ballot_sync(0xffffffffu, called), meths = __ballot_sync(0xffffffffu, is_m);
        if (!sites) continue;
        const uint32_t good[3] = {calls, meths, calls & ~meths};   // MHL: the sites that continue each family's run
        if (called) {
            uint32_t c = 0u, mm = 0u;
            if (ep.counts) last3(sites & below, calls, meths, c, mm);
            if (c == 7u || ep.mhl) {
                const uint32_t rank = cpg_rank(refcat, ep.rank, first_minus ? q - 1u : q);
                if (c == 7u) {
                    atomicAdd(ep.counts + (size_t)(rank - 3u) * 16 + ((mm << 1) | (is_m ? 1u : 0u)), 1u);
                    mine++;
                }
                if (ep.mhl) {
#pragma unroll
                    for (int t = 0; t < 2; t++) {
                        const int f = t == 0 ? 0 : (is_m ? 1 : 2);
                        const uint32_t mine_sites = sites & below, brk = mine_sites & ~good[f];
                        const uint32_t len = 1u + (brk ? (uint32_t)__popc(mine_sites >> (31 - __clz(brk))) - 1u : (uint32_t)__popc(mine_sites) + run[f]);
                        atomicAdd(ep.mhl + ((size_t)rank * 3 + f) * BSX_MHL_MAX_LEN + min(len, (uint32_t)BSX_MHL_MAX_LEN) - 1u, 1u);
                    }
                }
            }
        }
        if (ep.counts) {
            uint32_t c, mm;
            last3(sites, calls, meths, c, mm);
            c3 = c; m3 = mm;
        }
        if (ep.mhl) {
#pragma unroll
            for (int f = 0; f < 3; f++) {
                const uint32_t brk = sites & ~good[f];
                run[f] = min(brk ? (uint32_t)__popc(sites >> (31 - __clz(brk))) - 1u : run[f] + (uint32_t)__popc(sites), (uint32_t)BSX_MHL_MAX_LEN);
            }
            ncalls += (uint32_t)__popc(calls);
        }
    }
    mine = __reduce_add_sync(0xffffffffu, mine);
    if (lane == 0 && mine) { atomicAdd(&epi_count[0], 1u); atomicAdd(&epi_count[1], mine); }
    if (lane == 0 && ncalls) { atomicAdd(&mhl_count[0], 1u); atomicAdd(&mhl_count[1], ncalls); }
}

// One alignment, executed by a warp: get_alignment's trimming (methratio.py:56-64), the bounds test (105) and the
// pile-up (107-118).  getc(i) = i-th character of SEQ as printed.  Filters (-u / -p) were applied by the caller.
// Cycles: the call's cycle is its offset in printed SEQ, counted from the far end when SEQ is printed reversed (the two
// ZS characters differ); calls of read `read2` outside [5p, L - 3p) are dropped; the rest also go into `hist` (shared).
// Snp: a base over the complementary reference code counts into `confirm` (read G on '+' / C on '-') or `snp` (A / T),
// after the same trimming, bounds test and (Cycles) exclusion as a call.
// Conv (with Cycles): a first pass scores the alignment, its methylated calls whose context is not CpG, into conv_hist;
// an alignment scoring cv.threshold or more (when non-zero) returns before the second pass deposits anything.
// Pdr (with Cycles): the first pass also counts the methylated (pm) and unmethylated (pu) CpG calls; when the alignment is
// kept and pm + pu >= pd.min_cpg, the second pass adds each CpG call to pd.concordant (pm == 0 or pu == 0) or
// pd.discordant, and lane 0 counts the alignment in pdr_count (shared).
// Epi (with Cycles): the first pass also counts the CpG calls; with BSX_EPI_CPGS or more (MHL: one or more), a third
// pass (epi_windows) adds every fully called window of four consecutive sites to ep.counts and, with MHL, every call's
// runs to ep.mhl.
template <bool Cycles, bool Snp, bool Conv, bool Pdr, bool Epi, class GetC>
__device__ __forceinline__ void pile_alignment(const uint32_t *__restrict__ refcat, const uint32_t *__restrict__ seqinfo, uint32_t n_seq,
                                               uint32_t *meth, uint32_t *depth, unsigned long long *n_valid, const bsx_meth_opts &o,
                                               uint32_t k, long long pos, long long len, int st, int ins, long long mate_pos, bool sam, int lane, GetC getc,
                                               const MbiasArgs &mb = MbiasArgs{}, int read2 = 0, uint32_t *hist = nullptr,
                                               uint32_t *confirm = nullptr, uint32_t *snp = nullptr, const ConvArgs &cv = ConvArgs{},
                                               const PdrArgs &pd = PdrArgs{}, const EpiArgs &ep = EpiArgs{}) {
    const int L = (int)len;                                  // printed length, before trimming
    const uint32_t *anchor = seqinfo, *size = seqinfo + n_seq + 1;
    long long start = 0;
    const int N = o.trim_fillin;
    const bool first_minus = st & 1, second_minus = (st >> 1) & 1;
    if (N > 0) {                                             // trim fill-in nucleotides (methratio.py:56-63)
        if (!first_minus && second_minus) len = len - N > 0 ? len - N : 0;                     // '+-': seq[:-N]
        else if (first_minus && second_minus) { start = N < len ? N : len; len -= start; pos += N; }   // '--': seq[N:], pos + N
        else if (ins != 0 && len > (long long)abs(ins) - N) {
            const long long trim = len - ((long long)abs(ins) - N);
            if (!first_minus) len = len - trim > 0 ? len - trim : 0;                           // '++': seq[:-trim]
            else { start = trim < len ? trim : len; len -= start; pos += trim; }                // '-+': seq[trim:], pos + trim
        }
    }
    if (sam && ins > 0) {                                    // remove the region overlapped by the mate (methratio.py:64)
        const long long e = mate_pos - pos;                  // seq[:e] with Python slice semantics
        if (e < 0) len = len + e > 0 ? len + e : 0; else if (e < len) len = e;
    }
    if (pos + len > (long long)size[k]) return;             // methratio.py:105
    if (lane == 0) atomicAdd(n_valid, 1ull);
    const uint32_t base = anchor[k] + (uint32_t)pos;
    const uint32_t match = first_minus ? 2u : 1u;           // '+': C (converted reads show T), '-': G (A)
    const char cm = first_minus ? 'G' : 'C', cc = first_minus ? 'A' : 'T';
    const char ec = first_minus ? 'C' : 'G', es = first_minus ? 'T' : 'A';   // Snp: the opposite strand's base as printed
    if constexpr (!Cycles) {
        for (int i = lane; i < (int)len; i += 32) {
            const uint32_t r = ref_code(refcat, base + (uint32_t)i);
            if (r != match) {
                if constexpr (Snp) {
                    if (r == 3u - match) {
                        const char c = getc((int)start + i);
                        if (c == ec) atomicAdd(confirm + base + i, 1u);
                        else if (c == es) atomicAdd(snp + base + i, 1u);
                    }
                }
                continue;
            }
            const char c = getc((int)start + i);
            if (c == cc) atomicAdd(depth + base + i, 1u);
            else if (c == cm) { atomicAdd(meth + base + i, 1u); atomicAdd(depth + base + i, 1u); }
        }
    } else {
        const bool rev = ((st ^ (st >> 1)) & 1) != 0;
        const int lo = read2 ? mb.ignore[2] : mb.ignore[0], hi = L - (read2 ? mb.ignore[3] : mb.ignore[1]);
        uint32_t *pdr_to = nullptr;                          // Pdr: where the second pass adds the CpG calls; NULL = nowhere
        bool epi_walk = false;                               // Epi: the alignment has enough CpG calls for a window (MHL: one)
        if constexpr (Conv || Pdr || Epi) {
            // the score: a methylated call (read C on '+', G on '-') inside the cycle bounds whose next base on the call's
            // strand is not the CpG partner (CHG and CHH alike, so the second context code is not needed).  The bounds
            // [lo, hi) on the cycle are a range of i: cycle j = start + i, or L - 1 - j when reversed.  Pdr counts the
            // calls whose next base is the partner in the same loop, so it reads that base for unmethylated calls too.
            const int s0 = (int)start;
            const int i_end = min(rev ? L - s0 - lo : hi - s0, (int)len);
            uint32_t score = 0, pm = 0, pu = 0;
#pragma unroll 1
            for (int i = max(rev ? L - s0 - hi : lo - s0, 0) + lane; i < i_end; i += 32) {
                const uint32_t q = base + (uint32_t)i;
                if constexpr (!Pdr && !Epi) {
                    if (ref_code(refcat, q) != match || getc(s0 + i) != cm) continue;
                    const uint32_t c1 = first_minus ? ref_code(refcat, q - 1u) : ref_code(refcat, q + 1u);
                    score += c1 != 3u - match;
                } else {
                    if (ref_code(refcat, q) != match) continue;
                    const char c = getc(s0 + i);
                    const bool is_m = c == cm;
                    if (!is_m && c != cc) continue;
                    const uint32_t c1 = first_minus ? ref_code(refcat, q - 1u) : ref_code(refcat, q + 1u);
                    if (c1 == 3u - match) { pm += is_m; pu += !is_m; }
                    else if constexpr (Conv) score += is_m;
                }
            }
            if constexpr (Conv) {
                score = __reduce_add_sync(0xffffffffu, score);
                if (lane == 0) atomicAdd(&conv_hist[min(score, (uint32_t)BSX_CONV_BINS - 1u)], 1u);
                if (cv.threshold && score >= cv.threshold) return;
            }
            if constexpr (Pdr) {                             // the drop is decided, now the class
                pm = __reduce_add_sync(0xffffffffu, pm);
                pu = __reduce_add_sync(0xffffffffu, pu);
                if (pm + pu >= pd.min_cpg) {
                    const bool disc = pm != 0 && pu != 0;
                    pdr_to = disc ? pd.discordant : pd.concordant;
                    if (lane == 0) { atomicAdd(&pdr_count[0], 1u); if (disc) atomicAdd(&pdr_count[1], 1u); }
                }
            }
            if constexpr (Epi) epi_walk = (Pdr ? pm + pu : __reduce_add_sync(0xffffffffu, pm + pu)) >= (ep.mhl ? 1u : (uint32_t)BSX_EPI_CPGS);
        }
        uint32_t *h = hist + read2 * (3 * BSX_MBIAS_CYCLES * 2);
        for (int i = lane; i < (int)len; i += 32) {
            const uint32_t q = base + (uint32_t)i;
            const uint32_t r = ref_code(refcat, q);
            if (r != match) {
                if constexpr (Snp) {
                    if (r == 3u - match) {
                        const int j = (int)start + i;
                        const char c = getc(j);
                        uint32_t *ctr = c == ec ? confirm : (c == es ? snp : nullptr);
                        const int cyc = rev ? L - 1 - j : j;
                        if (ctr && cyc >= lo && cyc < hi) atomicAdd(ctr + q, 1u);
                    }
                }
                continue;
            }
            const int j = (int)start + i;
            const char c = getc(j);
            const bool is_m = c == cm;
            if (!is_m && c != cc) continue;
            const int cyc = rev ? L - 1 - j : j;
            if (cyc < lo || cyc >= hi) continue;
            atomicAdd(depth + q, 1u);
            if (is_m) atomicAdd(meth + q, 1u);
            // context on the call's strand: '+' looks at q+1, q+2 for G, '-' at q-1, q-2 for C; non-ACGT and the zero
            // margins / pads read as A, i.e. H
            const uint32_t want = 3u - match;
            const uint32_t c1 = first_minus ? ref_code(refcat, q - 1u) : ref_code(refcat, q + 1u);
            const uint32_t c2 = first_minus ? ref_code(refcat, q - 2u) : ref_code(refcat, q + 2u);
            const int ctx = c1 == want ? 0 : (c2 == want ? 1 : 2);
            if constexpr (Pdr) { if (pdr_to && ctx == 0) atomicAdd(pdr_to + q, 1u); }
            if (!mb.hist) continue;
            if (cyc < BSX_MBIAS_CYCLES) atomicAdd(h + (ctx * BSX_MBIAS_CYCLES + cyc) * 2 + (is_m ? 0 : 1), 1u);
            else atomicAdd(mb.hist + MBIAS_BINS, 1ull);
        }
        if constexpr (Epi) {
            if (epi_walk) epi_windows(refcat, base, (int)len, (int)start, L, rev, lo, hi, first_minus, match, cm, cc, lane, getc, ep);
        }
    }
}

// Cycles: a per-CTA histogram (M-bias; Conv: the scores), zeroed before and flushed (non-zero bins) after the CTA's
// alignments; out == NULL (exclusion without M-bias) skips both
template <int Bins>
__device__ __forceinline__ void hist_zero(uint32_t *hist, const unsigned long long *out) {
    if (!out) return;
    for (int b = threadIdx.x; b < Bins; b += blockDim.x) hist[b] = 0u;
    __syncthreads();
}
template <int Bins>
__device__ __forceinline__ void hist_flush(uint32_t *hist, unsigned long long *out) {
    if (!out) return;
    __syncthreads();
    for (int b = threadIdx.x; b < Bins; b += blockDim.x) { const uint32_t v = hist[b]; if (v) atomicAdd(out + b, (unsigned long long)v); }
}

// what get_alignment hands on (before trimming): sequence index, 0-based position, printed length, strand bits, ...
struct AlnView { uint32_t k; long long pos, len; int st, ins; long long mate_pos; bool sam; };

// -r key of an alignment (methratio.py:52-53): '+-' / '-+' hits are identified by where they end (direction 2), the
// others by where they start (direction 1).  A fragment end outside [0, size) makes the script raise IndexError (or
// wrap to the chromosome's last entry for -1); BSMAP never prints such a record, and here it skips the duplicate test.
__device__ __forceinline__ bool dup_key(const uint32_t *__restrict__ seqinfo, uint32_t n_seq, const AlnView &v, uint64_t &key) {
    const uint32_t *anchor = seqinfo, *size = seqinfo + n_seq + 1;
    const bool dir2 = ((v.st ^ (v.st >> 1)) & 1) != 0;
    const long long fe = dir2 ? v.pos + v.len : v.pos;
    if (fe < 0 || fe >= (long long)size[v.k]) return false;
    key = ((uint64_t)anchor[v.k] + (uint64_t)fe) * 2u + (dir2 ? 1u : 0u);
    return true;
}
// resolve (warp-uniform): does alignment `order` hold its key?  The holder marks it taken for every later batch.  A
// loser reads either the holder's claim or the 0 the holder has just written: both differ from its own claim.
__device__ __forceinline__ bool dup_holds(uint32_t *first, const uint32_t *__restrict__ seqinfo, uint32_t n_seq, const AlnView &v, uint32_t order, int lane) {
    uint64_t key;
    if (!dup_key(seqinfo, n_seq, v, key)) return true;
    uint32_t w = 0;
    if (lane == 0) { w = first[key]; if (w == order + 1u) first[key] = 0u; }
    w = __shfl_sync(0xffffffffu, w, 0);
    return w == order + 1u;
}

// alignment a of a batch parsed from SAM / BSP text on the host, after the -u / -p filters (methratio.py:35-36, 48-49)
__device__ __forceinline__ bool parsed_alignment(const bsx_meth_opts &o, uint32_t n_seq, uint32_t a, const uint16_t *__restrict__ lens,
                                                 const uint32_t *__restrict__ chr, const uint32_t *__restrict__ pos0, const uint8_t *__restrict__ strand,
                                                 const int32_t *__restrict__ insert, const int32_t *__restrict__ mate_pos, const uint8_t *__restrict__ flags, AlnView &v) {
    const uint32_t fl = flags[a];
    if (o.unique && (fl & BSX_METH_SECONDARY)) return false;
    if (o.pair && !(fl & BSX_METH_PROPER)) return false;
    v.k = chr[a];
    if (v.k >= n_seq) return false;
    v.pos = (long long)pos0[a]; v.len = (long long)lens[a]; v.st = strand[a]; v.ins = insert[a]; v.mate_pos = (long long)mate_pos[a];
    v.sam = (fl & BSX_METH_SAM) != 0;
    return true;
}

// -r, first kernel: one thread per alignment claims its key
__global__ void __launch_bounds__(256) meth_claim_kernel(const uint32_t *__restrict__ seqinfo, uint32_t n_seq, uint32_t *first, bsx_meth_opts o, uint32_t n,
                                                         const uint16_t *__restrict__ lens, const uint32_t *__restrict__ chr, const uint32_t *__restrict__ pos0,
                                                         const uint8_t *__restrict__ strand, const int32_t *__restrict__ insert,
                                                         const int32_t *__restrict__ mate_pos, const uint8_t *__restrict__ flags) {
    const uint32_t a = blockIdx.x * blockDim.x + threadIdx.x;
    AlnView v; uint64_t key;
    if (a < n && parsed_alignment(o, n_seq, a, lens, chr, pos0, strand, insert, mate_pos, flags, v) && dup_key(seqinfo, n_seq, v, key)) atomicMin(first + key, a + 1u);
}

// alignments parsed from SAM / BSP text on the host: one warp per alignment (Cycles: a grid-stride loop of them).
// Conv asks for 4 resident CTAs per SM: without that floor, ptxas squeezes its instantiations to 32 or 40 registers
// and spills; with it they take 38 - 44 and none.  Pdr and Epi take the same floor.  The other instantiations keep the
// plain bound (0 = none).
template <bool Cycles, bool Snp, bool Conv, bool Pdr, bool Epi>
__global__ void __launch_bounds__(256, (Conv || Pdr || Epi) ? 4 : 0) meth_pileup_kernel(const uint32_t *__restrict__ refcat, const uint32_t *__restrict__ seqinfo, uint32_t n_seq,
                                                          uint32_t *meth, uint32_t *depth, unsigned long long *n_valid, uint32_t *first, bsx_meth_opts o, uint32_t n,
                                                          const char *__restrict__ seqs, uint32_t stride, const uint16_t *__restrict__ lens,
                                                          const uint32_t *__restrict__ chr, const uint32_t *__restrict__ pos0,
                                                          const uint8_t *__restrict__ strand, const int32_t *__restrict__ insert,
                                                          const int32_t *__restrict__ mate_pos, const uint8_t *__restrict__ flags, MbiasArgs mb,
                                                          uint32_t *confirm, uint32_t *snp, ConvArgs cv, PdrArgs pd, EpiArgs ep) {
    static_assert(Cycles || !Conv, "the conversion filter runs in the Cycles kernels");
    static_assert(Cycles || !Pdr, "PDR runs in the Cycles kernels");
    static_assert(Cycles || !Epi, "epialleles run in the Cycles kernels");
    const uint32_t w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    auto one = [&](uint32_t a, uint32_t *hist) {
        AlnView v;
        if (!parsed_alignment(o, n_seq, a, lens, chr, pos0, strand, insert, mate_pos, flags, v)) return;
        if (first && !dup_holds(first, seqinfo, n_seq, v, a, lane)) return;
        const char *sq = seqs + (size_t)a * stride;
        pile_alignment<Cycles, Snp, Conv, Pdr, Epi>(refcat, seqinfo, n_seq, meth, depth, n_valid, o, v.k, v.pos, v.len, v.st, v.ins, v.mate_pos, v.sam, lane,
                                                    [sq](int i) { return sq[i]; }, mb, (flags[a] & BSX_METH_READ2) ? 1 : 0, hist, confirm, snp, cv, pd, ep);
    };
    if constexpr (!Cycles) {
        if (w >= n) return;
        one(w, nullptr);
    } else {
        __shared__ uint32_t hist[MBIAS_BINS];
        hist_zero<MBIAS_BINS>(hist, mb.hist);
        if constexpr (Conv) hist_zero<BSX_CONV_BINS>(conv_hist, cv.hist);
        if constexpr (Pdr) hist_zero<2>(pdr_count, pd.count);
        if constexpr (Epi) hist_zero<2>(epi_count, ep.count);
        if constexpr (Epi) hist_zero<2>(mhl_count, ep.mhl_count);
        for (uint32_t a = w; a < n; a += (gridDim.x * blockDim.x) >> 5) one(a, hist);
        hist_flush<MBIAS_BINS>(hist, mb.hist);
        if constexpr (Conv) hist_flush<BSX_CONV_BINS>(conv_hist, cv.hist);
        if constexpr (Pdr) hist_flush<2>(pdr_count, pd.count);
        if constexpr (Epi) hist_flush<2>(epi_count, ep.count);
        if constexpr (Epi) hist_flush<2>(mhl_count, ep.mhl_count);
    }
}

__device__ __forceinline__ char comp_char(char c) {   // rev_char[] (param.cpp:166-177)
    switch (c) {
        case 'A': return 'T'; case 'C': return 'G'; case 'G': return 'C'; case 'T': return 'A';
        case 'a': return 't'; case 'c': return 'g'; case 'g': return 'c'; case 't': return 'a';
        default: return 'N';
    }
}

// Unit u of the batch a mapper has just mapped (one read; PE: one mate), straight from its device buffers.  Which reads
// are printed as mapped, with which SEQ orientation / POS / TLEN / PNEXT, restates s_OutHit (align.cpp:631-765),
// s_OutHitPair (pairs.cpp:288-424) and s_OutHitUnpair (pairs.cpp:426-498); then the -u / -p filters.
__device__ __forceinline__ bool mapped_alignment(const bsx_meth_opts &o, int sam, int report_repeat_hits, uint32_t u, int mates,
                                                 const bsx_rec *__restrict__ out_a, const bsx_rec *__restrict__ out_b,
                                                 const bsx_pair_rec *__restrict__ out_pair, AlnView &v, bool &rev) {
    const uint32_t r = mates == 2 ? u >> 1 : u;
    const int mate = mates == 2 ? (int)(u & 1u) : 0;
    const bsx_rec rc = (mate ? out_b : out_a)[r];
    uint32_t chr, loc; int chain, lp = rc.len, ins = 0; long long mate_pos = -1; bool secondary, proper = false;
    if (mates == 2 && out_pair[r].paired) {
        const bsx_pair_rec pp = out_pair[r];
        const int la = out_a[r].len, lb = out_b[r].len;
        uint32_t a_loc = pp.a_loc, b_loc = pp.b_loc;
        // fragment shorter than the read: the adapter part is dropped (pairs.cpp:296-306)
        if (pp.insert < la && ((int)pp.chain ^ (int)(pp.a_chr & 1u))) a_loc += (uint32_t)(la - pp.insert);
        if (pp.insert < lb && ((!pp.chain) ^ (int)(pp.b_chr & 1u))) b_loc += (uint32_t)(lb - pp.insert);
        chr = mate ? pp.b_chr : pp.a_chr; loc = mate ? b_loc : a_loc; chain = mate ? !pp.chain : pp.chain;
        if (pp.insert < lp) lp = pp.insert;
        const bool rv = (chain ^ (int)(chr & 1u)) != 0;
        ins = sam ? (rv ? -pp.insert : pp.insert) : pp.insert;       // TLEN (pairs.cpp:330-340) / BSP insert column
        mate_pos = mate ? a_loc : b_loc;                             // PNEXT - 1
        secondary = pp.npairs > 1; proper = true;
    } else {
        const int nh = rc.status ? -1 : (int)rc.nhits;
        if (nh <= 0 || (nh > 1 && report_repeat_hits == 0)) return false;   // printed as unmapped ('u') or not at all
        chr = rc.chr; loc = rc.loc; chain = rc.chain; secondary = nh > 1;
    }
    if (o.unique && secondary) return false;
    if (o.pair && !proper) return false;
    rev = (chain ^ (int)(chr & 1u)) != 0;
    v.k = chr >> 1; v.pos = (long long)loc; v.len = (long long)lp; v.st = (int)(chr & 1u) | (chain << 1); v.ins = ins; v.mate_pos = mate_pos; v.sam = sam != 0;
    return true;
}

// -r, first kernel of the in-process form: one thread per unit claims its key (the order of the SAM lines: read by read, mate a before mate b)
__global__ void __launch_bounds__(256) meth_claim_mapped_kernel(const uint32_t *__restrict__ seqinfo, uint32_t n_seq, uint32_t *first, bsx_meth_opts o,
                                                                int sam, int report_repeat_hits, uint32_t n, int mates,
                                                                const bsx_rec *__restrict__ out_a, const bsx_rec *__restrict__ out_b,
                                                                const bsx_pair_rec *__restrict__ out_pair) {
    const uint32_t u = blockIdx.x * blockDim.x + threadIdx.x;
    AlnView v; bool rev; uint64_t key;
    if (u < n * (uint32_t)mates && mapped_alignment(o, sam, report_repeat_hits, u, mates, out_a, out_b, out_pair, v, rev) && dup_key(seqinfo, n_seq, v, key))
        atomicMin(first + key, u + 1u);
}

// pile-up of the mapped batch: one warp per read (PE: per mate; Cycles: a grid-stride loop of them); Conv's, Pdr's and
// Epi's bound as above
template <bool Cycles, bool Snp, bool Conv, bool Pdr, bool Epi>
__global__ void __launch_bounds__(256, (Conv || Pdr || Epi) ? 4 : 0) meth_pileup_mapped_kernel(const uint32_t *__restrict__ refcat, const uint32_t *__restrict__ seqinfo, uint32_t n_seq,
                                                                 uint32_t *meth, uint32_t *depth, unsigned long long *n_valid, uint32_t *first, bsx_meth_opts o,
                                                                 int sam, int report_repeat_hits, uint32_t n, int mates, uint32_t stride,
                                                                 const uint8_t *__restrict__ seq_a, const uint8_t *__restrict__ seq_b,
                                                                 const bsx_rec *__restrict__ out_a, const bsx_rec *__restrict__ out_b,
                                                                 const bsx_pair_rec *__restrict__ out_pair, MbiasArgs mb, uint32_t *confirm, uint32_t *snp,
                                                                 ConvArgs cv, PdrArgs pd, EpiArgs ep) {
    static_assert(Cycles || !Conv, "the conversion filter runs in the Cycles kernels");
    static_assert(Cycles || !Pdr, "PDR runs in the Cycles kernels");
    static_assert(Cycles || !Epi, "epialleles run in the Cycles kernels");
    const uint32_t w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    auto one = [&](uint32_t u, uint32_t *hist) {
        AlnView v; bool rev;
        if (!mapped_alignment(o, sam, report_repeat_hits, u, mates, out_a, out_b, out_pair, v, rev)) return;
        if (first && !dup_holds(first, seqinfo, n_seq, v, u, lane)) return;
        const uint32_t r = mates == 2 ? u >> 1 : u;
        const uint8_t *rd = ((mates == 2 && (u & 1u)) ? seq_b : seq_a) + (size_t)r * stride;
        const int lp = (int)v.len;
        const int read2 = mates == 2 ? (int)(u & 1u) : (mb.readset == 2 ? 1 : 0);     // mate b / readset 2 print FLAG 0x80
        pile_alignment<true, Snp, Conv, Pdr, Epi>(refcat, seqinfo, n_seq, meth, depth, n_valid, o, v.k, v.pos, v.len, v.st, v.ins, v.mate_pos, v.sam, lane,
                                                  [rd, rev, lp](int i) { return rev ? comp_char((char)rd[lp - 1 - i]) : (char)rd[i]; }, mb, read2, hist, confirm, snp,
                                                  cv, pd, ep);
    };
    if constexpr (!Cycles) {
        // the same steps as `one`, written out: through the lambda, ptxas allocates this instantiation differently
        const uint32_t u = w;
        if (u >= n * (uint32_t)mates) return;
        AlnView v; bool rev;
        if (!mapped_alignment(o, sam, report_repeat_hits, u, mates, out_a, out_b, out_pair, v, rev)) return;
        if (first && !dup_holds(first, seqinfo, n_seq, v, u, lane)) return;
        const uint32_t r = mates == 2 ? u >> 1 : u;
        const uint8_t *rd = ((mates == 2 && (u & 1u)) ? seq_b : seq_a) + (size_t)r * stride;
        const int lp = (int)v.len;
        pile_alignment<false, Snp, false, false, false>(refcat, seqinfo, n_seq, meth, depth, n_valid, o, v.k, v.pos, v.len, v.st, v.ins, v.mate_pos, v.sam, lane,
                                   [rd, rev, lp](int i) { return rev ? comp_char((char)rd[lp - 1 - i]) : (char)rd[i]; }, MbiasArgs{}, 0, nullptr, confirm, snp);
    } else {
        __shared__ uint32_t hist[MBIAS_BINS];
        hist_zero<MBIAS_BINS>(hist, mb.hist);
        if constexpr (Conv) hist_zero<BSX_CONV_BINS>(conv_hist, cv.hist);
        if constexpr (Pdr) hist_zero<2>(pdr_count, pd.count);
        if constexpr (Epi) hist_zero<2>(epi_count, ep.count);
        if constexpr (Epi) hist_zero<2>(mhl_count, ep.mhl_count);
        for (uint32_t u = w; u < n * (uint32_t)mates; u += (gridDim.x * blockDim.x) >> 5) one(u, hist);
        hist_flush<MBIAS_BINS>(hist, mb.hist);
        if constexpr (Conv) hist_flush<BSX_CONV_BINS>(conv_hist, cv.hist);
        if constexpr (Pdr) hist_flush<2>(pdr_count, pd.count);
        if constexpr (Epi) hist_flush<2>(epi_count, ep.count);
        if constexpr (Epi) hist_flush<2>(mhl_count, ep.mhl_count);
    }
}

// -g: every reference "CG": both counters of the C take the G's, the G's become 0 (methratio.py:122-131); Snp: the
// evidence counters the same way; Pdr: the concordance counters too
template <bool Snp, bool Pdr>
__global__ void meth_combine_kernel(const uint32_t *__restrict__ refcat, uint64_t n_pos, uint32_t *meth, uint32_t *depth, uint32_t *confirm, uint32_t *snp,
                                    uint32_t *conc, uint32_t *disc) {
    const uint64_t q = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q + 1 >= n_pos) return;
    if (ref_code(refcat, (uint32_t)q) == 1u && ref_code(refcat, (uint32_t)q + 1u) == 2u) {
        depth[q] += depth[q + 1]; meth[q] += meth[q + 1];
        depth[q + 1] = 0; meth[q + 1] = 0;
        if constexpr (Snp) {
            confirm[q] += confirm[q + 1]; snp[q] += snp[q + 1];
            confirm[q + 1] = 0; snp[q + 1] = 0;
        }
        if constexpr (Pdr) {
            conc[q] += conc[q + 1]; disc[q] += disc[q + 1];
            conc[q + 1] = 0; disc[q + 1] = 0;
        }
    }
}

// Region reduction (bsx_meth_regions).  Every region is cut into chunks of REGION_CHUNK positions; scan[r] is the
// exclusive sum of chunks over the regions before r (scan[n] = all), so a warp takes one chunk whatever the regions'
// sizes.  4096 positions = 128 per lane: the 12 atomics and the reduction of a chunk cost little next to its 32 KB of
// counters, and a 1 kb tile is still one chunk.
constexpr uint32_t REGION_CHUNK = 4096;
constexpr uint64_t REGION_SLICE = 1u << 20;     // regions per launch: bounds the device buffers (scan, spans, 96 MB of sums)

// One warp per chunk (a grid-stride loop of them).  Lanes read meth / depth (and the evidence the mode needs)
// coalesced, and the reference codes q-2..q+2 from two refcat words; the pads between sequences are zero (A), so
// positions off the sequence read as H.  Per lane: sites, covered, C and CT of the three contexts in registers, reduced
// over the warp, then lanes 0-11 add them to out[(r * 3 + ctx) * 4 + {sites, covered, C, CT}] (u64: exact, and
// independent of the schedule).  Combine: -g's site rule (a G after a C is no site).  Snp: BSX_CT_SNP_SKIP drops a
// covered site with any SNP evidence, BSX_CT_SNP_CORRECT one whose SNP-corrected depth is 0; 0 = no drop rule.
// Pdr: also the sums of conc and disc over the positions the PDR file prints (conc + disc >= min_depth, the same drop
// rule), which lane 0 adds to pdr_out[r * 2 + {0, 1}].
template <bool Combine, int Snp, bool Pdr>
__global__ void __launch_bounds__(256) meth_region_kernel(const uint32_t *__restrict__ refcat, const uint32_t *__restrict__ meth,
                                                          const uint32_t *__restrict__ depth, const uint32_t *__restrict__ confirm,
                                                          const uint32_t *__restrict__ snp, uint32_t min_depth,
                                                          const unsigned long long *__restrict__ scan, const uint2 *__restrict__ span, uint32_t n,
                                                          unsigned long long *out, const uint32_t *__restrict__ conc,
                                                          const uint32_t *__restrict__ disc, unsigned long long *pdr_out) {
    const int lane = threadIdx.x & 31;
    const unsigned long long total = scan[n], warps = ((unsigned long long)gridDim.x * blockDim.x) >> 5;
    for (unsigned long long c = ((unsigned long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; c < total; c += warps) {
        // the chunk's region: the last r with scan[r] <= c, by a 32-way search (scan[lo] <= c < scan[hi] throughout)
        uint32_t lo = 0, hi = n;
        while (hi - lo > 1) {
            const uint32_t step = (hi - lo + 31) / 32, idx = lo + (uint32_t)lane * step;
            const unsigned ball = __ballot_sync(0xffffffffu, idx < hi && scan[idx] <= c);
            lo += (uint32_t)(31 - __clz(ball)) * step;
            hi = min(hi, lo + step);
        }
        const uint2 s = span[lo];
        const uint32_t b = s.x + (uint32_t)(c - scan[lo]) * REGION_CHUNK, e = min(b + REGION_CHUNK, s.y);
        uint32_t sites[3] = {0u, 0u, 0u}, cov[3] = {0u, 0u, 0u};
        unsigned long long cm[3] = {0ull, 0ull, 0ull}, ct[3] = {0ull, 0ull, 0ull};
        unsigned long long pc = 0, pdd = 0;
        for (uint32_t q = b + (uint32_t)lane; q < e; q += 32) {
            const uint32_t a = (q - 2u) >> 4, sh = (q - 2u) & 15u;     // bases q-2 .. q+2 lie in words a, a+1
            const unsigned long long w = ((unsigned long long)__ldg(refcat + a) << 32) | __ldg(refcat + a + 1);
            auto code = [&](uint32_t k) { return (uint32_t)(w >> (62u - 2u * (sh + k))) & 3u; };
            const uint32_t r = code(2), before = code(1);
            const bool plus = r == 1u;
            bool site = plus || r == 2u;
            if constexpr (Combine) site = site && !(r == 2u && before == 1u);
            const uint32_t want = plus ? 2u : 1u, c1 = plus ? code(3) : before, c2 = plus ? code(4) : code(0);
            const int ctx = c1 == want ? 0 : (c2 == want ? 1 : 2);
            const uint32_t d = depth[q], mm = meth[q];
            bool covered = site && d >= min_depth;
            if constexpr (Snp == BSX_CT_SNP_SKIP) covered = covered && snp[q] == 0u;
            if constexpr (Snp == BSX_CT_SNP_CORRECT) covered = covered && (snp[q] == 0u || confirm[q] != 0u);
#pragma unroll
            for (int k = 0; k < 3; k++) {
                const bool in = ctx == k;
                sites[k] += (site && in) ? 1u : 0u;
                if (covered && in) { cov[k] += 1u; cm[k] += mm; ct[k] += d; }
            }
            if constexpr (Pdr) {
                const unsigned long long x = conc[q], y = disc[q];
                bool shown = x + y >= min_depth;
                if constexpr (Snp == BSX_CT_SNP_SKIP) shown = shown && snp[q] == 0u;
                if constexpr (Snp == BSX_CT_SNP_CORRECT) shown = shown && (snp[q] == 0u || confirm[q] != 0u);
                if (shown) { pc += x; pdd += y; }
            }
        }
#pragma unroll
        for (int k = 0; k < 3; k++) {
            sites[k] = __reduce_add_sync(0xffffffffu, sites[k]);
            cov[k] = __reduce_add_sync(0xffffffffu, cov[k]);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) { cm[k] += __shfl_xor_sync(0xffffffffu, cm[k], o); ct[k] += __shfl_xor_sync(0xffffffffu, ct[k], o); }
        }
        unsigned long long v = 0;
#pragma unroll
        for (int k = 0; k < 3; k++) {
            if (lane == 4 * k) v = sites[k];
            if (lane == 4 * k + 1) v = cov[k];
            if (lane == 4 * k + 2) v = cm[k];
            if (lane == 4 * k + 3) v = ct[k];
        }
        if (lane < 12 && v) atomicAdd(out + (size_t)lo * 12 + lane, v);
        if constexpr (Pdr) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) { pc += __shfl_xor_sync(0xffffffffu, pc, o); pdd += __shfl_xor_sync(0xffffffffu, pdd, o); }
            if (lane == 0 && pc) atomicAdd(pdr_out + (size_t)lo * 2, pc);
            if (lane == 0 && pdd) atomicAdd(pdr_out + (size_t)lo * 2 + 1, pdd);
        }
    }
}

template <bool Pdr>
auto region_kernel_of(bool combine, int snp_mode) {
    if (snp_mode == BSX_CT_SNP_SKIP) return combine ? meth_region_kernel<true, BSX_CT_SNP_SKIP, Pdr> : meth_region_kernel<false, BSX_CT_SNP_SKIP, Pdr>;
    if (snp_mode == BSX_CT_SNP_CORRECT) return combine ? meth_region_kernel<true, BSX_CT_SNP_CORRECT, Pdr> : meth_region_kernel<false, BSX_CT_SNP_CORRECT, Pdr>;
    return combine ? meth_region_kernel<true, 0, Pdr> : meth_region_kernel<false, 0, Pdr>;
}
auto region_kernel(bool combine, int snp_mode, bool pdr) { return pdr ? region_kernel_of<true>(combine, snp_mode) : region_kernel_of<false>(combine, snp_mode); }

// MHL's region reduction (bsx_meth_regions_mhl).  A region's sites are a rank range [a, b); it is cut into chunks of
// MHL_CHUNK ranks, and scan[r] is the exclusive sum of chunks over the regions before r, as for meth_region_kernel.  A
// slice of regions takes 48 u64 sums each, so it holds a quarter of REGION_SLICE's regions (96 MB of sums again).
constexpr uint32_t MHL_CHUNK = 256;
constexpr uint64_t MHL_SLICE = REGION_SLICE / 4;

// the rank of the first site at or after position c (c may be the end of the packed reference: then no word is read)
__device__ __forceinline__ uint32_t cpg_rank_at(const uint32_t *__restrict__ refcat, const uint32_t *__restrict__ rank, uint32_t c) {
    return (c & 15u) ? cpg_rank(refcat, rank, c) : __ldg(rank + (c >> 4));
}

// one thread per region: its rank range from its clipped positions, and its chunks (chunks[n] = 0 ends the scan)
__global__ void __launch_bounds__(256) mhl_span_kernel(const uint32_t *__restrict__ refcat, const uint32_t *__restrict__ rank,
                                                       const uint2 *__restrict__ pos, uint32_t n, uint2 *span, uint32_t *chunks) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i > n) return;
    if (i == n) { chunks[n] = 0u; return; }
    const uint2 p = pos[i];
    const uint32_t a = cpg_rank_at(refcat, rank, p.x), b = cpg_rank_at(refcat, rank, p.y);
    span[i] = make_uint2(a, b);
    chunks[i] = (b - a + MHL_CHUNK - 1) / MHL_CHUNK;
}

// the SNP modes' cut sites: bit s of cut set when site s has SNP evidence (snp > 0) at its C or its G.  One thread per
// packed word; its sites, in ascending rank.
__global__ void __launch_bounds__(256) mhl_cut_kernel(const uint32_t *__restrict__ refcat, uint64_t n_words, const uint32_t *__restrict__ rank,
                                                      const uint32_t *__restrict__ snp, uint32_t *cut) {
    const uint64_t a = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (a >= n_words) return;
    uint32_t s = cpg_mask(refcat[a], a + 1 < n_words ? refcat[a + 1] : 0u), r = rank[a];
    while (s) {
        const int b = 31 - __clz(s);
        s &= ~(1u << b);
        const uint64_t c = a * 16 + (uint64_t)((30 - b) >> 1);
        if (snp[c] || snp[c + 1]) atomicOr(cut + (r >> 5), 1u << (r & 31u));
        r++;
    }
}

// One warp per chunk (a grid-stride loop of them), two sites a step: lanes 0-15 take site s, 16-31 site s + 1, lane
// l - 1 of each half the run length r = l.  Per family, the half's 16 counters are summed over r >= l (a suffix sum by
// shuffles; in u32, as it is bounded by the alignments with a call at the site, which the u32 depth counter also
// counts), and added to the lane's T_l / M_l / U_l while l <= lim: the region's sites up to s and, with cuts, those
// since the last cut (0 at a cut site), capped at 16, carried warp-uniformly from site to site.  The halves are added
// and lanes 0-15 add the 48 sums to out[(r * 3 + f) * 16 + l - 1] (u64 atomics: exact and independent of the schedule).
__global__ void __launch_bounds__(256) meth_mhl_region_kernel(const uint32_t *__restrict__ counts, const uint32_t *__restrict__ cut,
                                                              const uint32_t *__restrict__ scan, const uint2 *__restrict__ span, uint32_t n,
                                                              unsigned long long *out) {
    const int lane = threadIdx.x & 31, half = lane >> 4, l1 = lane & 15;
    const uint32_t total = scan[n], warps = (gridDim.x * blockDim.x) >> 5;
    auto is_cut = [&](uint32_t s) { return cut && ((__ldg(cut + (s >> 5)) >> (s & 31u)) & 1u); };
    for (uint32_t c = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; c < total; c += warps) {
        uint32_t lo = 0, hi = n;                                // the chunk's region, as in meth_region_kernel
        while (hi - lo > 1) {
            const uint32_t step = (hi - lo + 31) / 32, idx = lo + (uint32_t)lane * step;
            const unsigned ball = __ballot_sync(0xffffffffu, idx < hi && scan[idx] <= c);
            lo += (uint32_t)(31 - __clz(ball)) * step;
            hi = min(hi, lo + step);
        }
        const uint2 sp = span[lo];
        const uint32_t b = sp.x + (c - scan[lo]) * MHL_CHUNK, e = min(b + MHL_CHUNK, sp.y);
        uint32_t run = min(b - sp.x, (uint32_t)BSX_MHL_MAX_LEN);  // lim of site b - 1
        for (uint32_t t = 1; t <= run; t++) if (is_cut(b - t)) { run = t - 1; break; }
        unsigned long long acc[3] = {0ull, 0ull, 0ull};
        for (uint32_t s0 = b; s0 < e; s0 += 2) {
            const uint32_t r0 = is_cut(s0) ? 0u : min(run + 1u, (uint32_t)BSX_MHL_MAX_LEN);
            const bool two = s0 + 1 < e;
            const uint32_t r1 = (!two || is_cut(s0 + 1)) ? 0u : min(r0 + 1u, (uint32_t)BSX_MHL_MAX_LEN);
            run = two ? r1 : r0;
            const uint32_t lim = half ? r1 : r0;
            const uint32_t *row = counts + (size_t)(s0 + (uint32_t)half) * (3 * BSX_MHL_MAX_LEN) + l1;
#pragma unroll
            for (int f = 0; f < 3; f++) {
                uint32_t v = lim ? __ldg(row + f * BSX_MHL_MAX_LEN) : 0u;
#pragma unroll
                for (int o = 1; o < 16; o <<= 1) {
                    const uint32_t y = __shfl_down_sync(0xffffffffu, v, o, 16);
                    if (l1 + o < 16) v += y;
                }
                if ((uint32_t)l1 < lim) acc[f] += v;
            }
        }
#pragma unroll
        for (int f = 0; f < 3; f++) {
            acc[f] += __shfl_xor_sync(0xffffffffu, acc[f], 16);
            if (lane < 16 && acc[f]) atomicAdd(out + ((size_t)lo * 3 + f) * BSX_MHL_MAX_LEN + l1, acc[f]);
        }
    }
}

// Epi's rank index, first step: the CpG sites of each packed word (x[n_words] = 0, so that the scan ends in the total)
__global__ void __launch_bounds__(256) cpg_count_kernel(const uint32_t *__restrict__ refcat, uint64_t n_words, uint32_t *x) {
    const uint64_t a = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (a > n_words) return;
    x[a] = a < n_words ? (uint32_t)__popc(cpg_mask(refcat[a], a + 1 < n_words ? refcat[a + 1] : 0u)) : 0u;
}

// exclusive scan of u32 in place: each CTA scans a tile of SCAN_TILE (8 per thread, then the warps, then the CTA's 8
// warp sums) and writes the tile's total to sums; the tiles' totals are scanned the same way (recursively) and added
constexpr int SCAN_TILE = 256 * 8;
__global__ void __launch_bounds__(256) scan_tile_kernel(uint32_t *x, uint64_t n, uint32_t *sums) {
    __shared__ uint32_t warp_sum[8];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint64_t b = (uint64_t)blockIdx.x * SCAN_TILE + (uint64_t)threadIdx.x * 8;
    uint32_t v[8], t = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) { const uint32_t y = b + k < n ? x[b + k] : 0u; v[k] = t; t += y; }
    uint32_t inc = t;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const uint32_t y = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += y; }
    if (lane == 31) warp_sum[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        uint32_t w = lane < 8 ? warp_sum[lane] : 0u, wi = w;
#pragma unroll
        for (int o = 1; o < 8; o <<= 1) { const uint32_t y = __shfl_up_sync(0xffffffffu, wi, o); if (lane >= o) wi += y; }
        __syncwarp();
        if (lane < 8) warp_sum[lane] = wi - w;
    }
    __syncthreads();
    const uint32_t off = warp_sum[warp] + inc - t;
#pragma unroll
    for (int k = 0; k < 8; k++) if (b + k < n) x[b + k] = v[k] + off;
    if (threadIdx.x == blockDim.x - 1) sums[blockIdx.x] = off + t;
}
__global__ void __launch_bounds__(256) scan_add_kernel(uint32_t *x, uint64_t n, const uint32_t *__restrict__ tile_off) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) x[i] += tile_off[i / SCAN_TILE];
}
int scan_exclusive(uint32_t *x, uint64_t n) {
    const uint64_t tiles = (n + SCAN_TILE - 1) / SCAN_TILE;
    uint32_t *sums = nullptr;
    if (cudaMalloc(&sums, tiles * 4) != cudaSuccess) { cudaGetLastError(); bsx_set_error("epialleles: out of device memory (%llu bytes for the scan)", (unsigned long long)tiles * 4); return BSX_ERR_CUDA; }
    scan_tile_kernel<<<(unsigned)tiles, 256>>>(x, n, sums);
    int rc = cudaGetLastError() == cudaSuccess ? BSX_OK : BSX_ERR_CUDA;
    if (rc) bsx_set_error("epialleles: scan kernel failed");
    if (!rc && tiles > 1) rc = scan_exclusive(sums, tiles);
    if (!rc && tiles > 1) {
        scan_add_kernel<<<(unsigned)((n + 255) / 256), 256>>>(x, n, sums);
        if (cudaGetLastError() != cudaSuccess) { bsx_set_error("epialleles: scan kernel failed"); rc = BSX_ERR_CUDA; }
    }
    cudaDeviceSynchronize();
    cudaFree(sums);
    return rc;
}

// the CpG rank index, built once for epialleles and MHL; `what` names the option in messages
int ensure_cpg_rank(bsx_meth *m, const char *what) {
    if (m->d_cpg_rank) return BSX_OK;
    const uint64_t nw = m->ix->n_words;
    if (cudaMalloc(&m->d_cpg_rank, (nw + 1) * 4) != cudaSuccess) {
        cudaGetLastError(); m->d_cpg_rank = nullptr;
        bsx_set_error("%s: out of device memory (%llu bytes for the CpG rank index)", what, (unsigned long long)(nw + 1) * 4); return BSX_ERR_CUDA; }
    auto undo = [m]() { cudaFree(m->d_cpg_rank); m->d_cpg_rank = nullptr; };
    cpg_count_kernel<<<(unsigned)((nw + 1 + 255) / 256), 256>>>(m->ix->d_refcat, nw, m->d_cpg_rank);
    if (cudaGetLastError() != cudaSuccess) { undo(); bsx_set_error("%s: CpG count kernel failed", what); return BSX_ERR_CUDA; }
    const int rc = scan_exclusive(m->d_cpg_rank, nw + 1);
    if (rc) { undo(); return rc; }
    uint32_t sites = 0;
    if (cudaMemcpy(&sites, m->d_cpg_rank + nw, 4, cudaMemcpyDeviceToHost) != cudaSuccess) { cudaGetLastError(); undo(); bsx_set_error("%s: rank index download failed", what); return BSX_ERR_CUDA; }
    m->cpg_sites = sites;
    return BSX_OK;
}

int ensure_staging(bsx_meth *m, size_t n, uint32_t stride) {
    if (n <= m->cap && stride <= m->stride) return BSX_OK;
    cudaFree(m->d_seq); cudaFree(m->d_len); cudaFree(m->d_chr); cudaFree(m->d_pos); cudaFree(m->d_strand); cudaFree(m->d_flags); cudaFree(m->d_ins); cudaFree(m->d_mate);
    m->cap = std::max(n, m->cap); m->stride = std::max(stride, m->stride);
    BSX_CUDA_CHECK(cudaMalloc(&m->d_seq, m->cap * m->stride));
    BSX_CUDA_CHECK(cudaMalloc(&m->d_len, m->cap * 2));
    BSX_CUDA_CHECK(cudaMalloc(&m->d_chr, m->cap * 4));
    BSX_CUDA_CHECK(cudaMalloc(&m->d_pos, m->cap * 4));
    BSX_CUDA_CHECK(cudaMalloc(&m->d_strand, m->cap));
    BSX_CUDA_CHECK(cudaMalloc(&m->d_flags, m->cap));
    BSX_CUDA_CHECK(cudaMalloc(&m->d_ins, m->cap * 4));
    BSX_CUDA_CHECK(cudaMalloc(&m->d_mate, m->cap * 4));
    return BSX_OK;
}

// -r: the claim table, all keys free
int ensure_dup_table(bsx_meth *m) {
    if (m->d_first) return BSX_OK;
    const size_t bytes = m->ix->n_words * 16 * 2 * sizeof(uint32_t);
    if (cudaMalloc(&m->d_first, bytes) != cudaSuccess) { cudaGetLastError(); bsx_set_error("-r: out of device memory (%zu bytes for the duplicate table)", bytes); return BSX_ERR_CUDA; }
    BSX_CUDA_CHECK(cudaMemset(m->d_first, 0xff, bytes));
    BSX_CUDA_CHECK(cudaEventCreateWithFlags(&m->dup_order, cudaEventDisableTiming));
    BSX_CUDA_CHECK(cudaDeviceSynchronize());
    return BSX_OK;
}

// the instantiation for a combination of options (the kernels of one combination share a signature); conv, pdr and epi
// imply cycles
auto text_kernel(bool cycles, bool snp, bool conv, bool pdr, bool epi) {
    if (epi) return pdr ? (conv ? (snp ? meth_pileup_kernel<true, true, true, true, true> : meth_pileup_kernel<true, false, true, true, true>)
                                : (snp ? meth_pileup_kernel<true, true, false, true, true> : meth_pileup_kernel<true, false, false, true, true>))
                        : (conv ? (snp ? meth_pileup_kernel<true, true, true, false, true> : meth_pileup_kernel<true, false, true, false, true>)
                                : (snp ? meth_pileup_kernel<true, true, false, false, true> : meth_pileup_kernel<true, false, false, false, true>));
    if (pdr) return conv ? (snp ? meth_pileup_kernel<true, true, true, true, false> : meth_pileup_kernel<true, false, true, true, false>)
                         : (snp ? meth_pileup_kernel<true, true, false, true, false> : meth_pileup_kernel<true, false, false, true, false>);
    if (conv) return snp ? meth_pileup_kernel<true, true, true, false, false> : meth_pileup_kernel<true, false, true, false, false>;
    return cycles ? (snp ? meth_pileup_kernel<true, true, false, false, false> : meth_pileup_kernel<true, false, false, false, false>)
                  : (snp ? meth_pileup_kernel<false, true, false, false, false> : meth_pileup_kernel<false, false, false, false, false>);
}
auto mapped_kernel(bool cycles, bool snp, bool conv, bool pdr, bool epi) {
    if (epi) return pdr ? (conv ? (snp ? meth_pileup_mapped_kernel<true, true, true, true, true> : meth_pileup_mapped_kernel<true, false, true, true, true>)
                                : (snp ? meth_pileup_mapped_kernel<true, true, false, true, true> : meth_pileup_mapped_kernel<true, false, false, true, true>))
                        : (conv ? (snp ? meth_pileup_mapped_kernel<true, true, true, false, true> : meth_pileup_mapped_kernel<true, false, true, false, true>)
                                : (snp ? meth_pileup_mapped_kernel<true, true, false, false, true> : meth_pileup_mapped_kernel<true, false, false, false, true>));
    if (pdr) return conv ? (snp ? meth_pileup_mapped_kernel<true, true, true, true, false> : meth_pileup_mapped_kernel<true, false, true, true, false>)
                         : (snp ? meth_pileup_mapped_kernel<true, true, false, true, false> : meth_pileup_mapped_kernel<true, false, false, true, false>);
    if (conv) return snp ? meth_pileup_mapped_kernel<true, true, true, false, false> : meth_pileup_mapped_kernel<true, false, true, false, false>;
    return cycles ? (snp ? meth_pileup_mapped_kernel<true, true, false, false, false> : meth_pileup_mapped_kernel<true, false, false, false, false>)
                  : (snp ? meth_pileup_mapped_kernel<false, true, false, false, false> : meth_pileup_mapped_kernel<false, false, false, false, false>);
}

// the Cycles kernels run for M-bias, exclusion, the conversion filter, PDR, epialleles or MHL (with M-bias and exclusion off,
// Cycles is the classification alone: no histogram, bounds [0, L))
bool cycles_on(const bsx_meth *m) {
    return m->mbias || m->ignore[0] || m->ignore[1] || m->ignore[2] || m->ignore[3] || m->d_conv || m->d_pdr || m->d_epi || m->d_mhl;
}
// the Epi instantiation serves epialleles, MHL or both
bool epi_on(const bsx_meth *m) { return m->d_epi || m->d_mhl; }

// the Cycles kernels' grid cap and, with M-bias on, their histogram (zeroed), on the first pile-up that needs them
int ensure_cycles(bsx_meth *m) {
    if (m->resident[0]) return BSX_OK;
    if (m->mbias) {
        BSX_CUDA_CHECK(cudaMalloc(&m->d_mbias, (MBIAS_BINS + 1) * sizeof(unsigned long long)));
        BSX_CUDA_CHECK(cudaMemset(m->d_mbias, 0, (MBIAS_BINS + 1) * sizeof(unsigned long long)));
    }
    int dev = 0, sms = 0, per_sm[2] = {0, 0};
    BSX_CUDA_CHECK(cudaGetDevice(&dev));
    BSX_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    BSX_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm[0], text_kernel(true, m->ct_snp != 0, m->d_conv != nullptr, m->d_pdr != nullptr, epi_on(m)), 256, 0));
    BSX_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm[1], mapped_kernel(true, m->ct_snp != 0, m->d_conv != nullptr, m->d_pdr != nullptr, epi_on(m)), 256, 0));
    for (int i = 0; i < 2; i++) m->resident[i] = std::max(per_sm[i], 1) * sms;
    BSX_CUDA_CHECK(cudaDeviceSynchronize());
    return BSX_OK;
}
MbiasArgs mbias_args(const bsx_meth *m, int readset) {
    MbiasArgs a{};
    a.hist = m->d_mbias; a.readset = readset;          // NULL without M-bias: the kernels keep no histogram
    for (int i = 0; i < 4; i++) a.ignore[i] = m->ignore[i];
    return a;
}
ConvArgs conv_args(const bsx_meth *m) { return ConvArgs{m->d_conv, (uint32_t)m->conv_threshold}; }
PdrArgs pdr_args(const bsx_meth *m) { return PdrArgs{m->d_conc, m->d_disc, m->d_pdr, m->pdr_min_cpg}; }
EpiArgs epi_args(const bsx_meth *m) { return EpiArgs{m->d_cpg_rank, m->d_epi, m->d_epi_count, m->d_mhl, m->d_mhl_count}; }

int combine_once(bsx_meth *m, const bsx_meth_opts *o) {
    if (!o->combine_cpg || m->combined) return BSX_OK;
    const uint64_t n_pos = m->ix->n_words * 16;
    const auto kern = m->d_pdr ? (m->ct_snp ? meth_combine_kernel<true, true> : meth_combine_kernel<false, true>)
                               : (m->ct_snp ? meth_combine_kernel<true, false> : meth_combine_kernel<false, false>);
    kern<<<(unsigned)((n_pos + 255) / 256), 256>>>(m->ix->d_refcat, n_pos, m->d_meth, m->d_depth, m->d_confirm, m->d_snp, m->d_conc, m->d_disc);
    BSX_CUDA_CHECK(cudaGetLastError());
    BSX_CUDA_CHECK(cudaDeviceSynchronize());
    m->combined = true;
    return BSX_OK;
}

struct Sink {
    std::string *s;
    void put(const char *p, size_t n) { s->append(p, n); }
    void putc(char c) { s->push_back(c); }
    void putu(unsigned long long v) { char b[24]; char *e = b + 24, *q = e; do { *--q = (char)('0' + v % 10); v /= 10; } while (v); put(q, (size_t)(e - q)); }
    void putf3(double v) { char b[48]; const int l = snprintf(b, sizeof b, "%.3f", v); put(b, (size_t)l); }
    void putf2(double v) { char b[48]; const int l = snprintf(b, sizeof b, "%.2f", v); put(b, (size_t)l); }
    void putf4(double v) { char b[48]; const int l = snprintf(b, sizeof b, "%.4f", v); put(b, (size_t)l); }
};

}  // namespace

extern "C" void bsx_meth_opts_default(bsx_meth_opts *o) {
    if (!o) return;
    memset(o, 0, sizeof *o);
    o->trim_fillin = 2; o->min_depth = 1;
}

extern "C" int bsx_meth_create(const bsx_index *ix, bsx_meth **out) {
    if (!ix || !out) { bsx_set_error("bsx_meth_create: bad argument"); return BSX_ERR_ARG; }
    if (ix->device < 0) { bsx_set_error("text-only index has no device arrays: methratio needs the index on a CUDA device"); return BSX_ERR_CUDA; }
    BSX_CUDA_CHECK(cudaSetDevice(ix->device));
    bsx_meth *m = new bsx_meth();
    m->ix = ix;
    const size_t bytes = ix->n_words * 16 * sizeof(uint32_t);
    if (cudaMalloc(&m->d_meth, bytes) != cudaSuccess || cudaMalloc(&m->d_depth, bytes) != cudaSuccess || cudaMalloc(&m->d_valid, 8) != cudaSuccess) {
        cudaGetLastError(); bsx_meth_destroy(m); bsx_set_error("bsx_meth_create: out of device memory (%zu bytes per counter array)", bytes); return BSX_ERR_CUDA; }
    BSX_CUDA_CHECK(cudaMemset(m->d_meth, 0, bytes));
    BSX_CUDA_CHECK(cudaMemset(m->d_depth, 0, bytes));
    BSX_CUDA_CHECK(cudaMemset(m->d_valid, 0, 8));
    *out = m;
    return BSX_OK;
}

extern "C" int bsx_meth_destroy(bsx_meth *m) {
    if (!m) return BSX_OK;
    cudaFree(m->d_meth); cudaFree(m->d_depth); cudaFree(m->d_valid); cudaFree(m->d_first); cudaFree(m->d_mbias); cudaFree(m->d_confirm); cudaFree(m->d_snp); cudaFree(m->d_conv);
    cudaFree(m->d_conc); cudaFree(m->d_disc); cudaFree(m->d_pdr); cudaFree(m->d_cpg_rank); cudaFree(m->d_epi); cudaFree(m->d_epi_count);
    cudaFree(m->d_mhl); cudaFree(m->d_mhl_count);
    if (m->dup_order) cudaEventDestroy(m->dup_order);
    cudaFree(m->d_seq); cudaFree(m->d_len); cudaFree(m->d_chr); cudaFree(m->d_pos); cudaFree(m->d_strand); cudaFree(m->d_flags); cudaFree(m->d_ins); cudaFree(m->d_mate);
    delete m;
    return BSX_OK;
}

extern "C" int bsx_meth_add(bsx_meth *m, const bsx_meth_opts *o, uint32_t n, const char *seqs, uint32_t stride,
                            const uint16_t *lens, const uint32_t *chr, const uint32_t *pos, const uint8_t *strand,
                            const int32_t *insert, const int32_t *mate_pos, const uint8_t *flags, uint64_t *n_valid) {
    if (!m || !o || (n && (!seqs || !lens || !chr || !pos || !strand || !insert || !mate_pos || !flags))) { bsx_set_error("bsx_meth_add: bad argument"); return BSX_ERR_ARG; }
    if (m->combined) { bsx_set_error("bsx_meth_add: counters were already combined (-g); create a new bsx_meth"); return BSX_ERR_ARG; }
    BSX_CUDA_CHECK(cudaSetDevice(m->ix->device));
    if (n) {
        m->started = true;
        int rc = ensure_staging(m, n, stride); if (rc) return rc;
        BSX_CUDA_CHECK(cudaMemcpy2D(m->d_seq, m->stride, seqs, stride, stride, n, cudaMemcpyHostToDevice));
        BSX_CUDA_CHECK(cudaMemcpy(m->d_len, lens, (size_t)n * 2, cudaMemcpyHostToDevice));
        BSX_CUDA_CHECK(cudaMemcpy(m->d_chr, chr, (size_t)n * 4, cudaMemcpyHostToDevice));
        BSX_CUDA_CHECK(cudaMemcpy(m->d_pos, pos, (size_t)n * 4, cudaMemcpyHostToDevice));
        BSX_CUDA_CHECK(cudaMemcpy(m->d_strand, strand, n, cudaMemcpyHostToDevice));
        BSX_CUDA_CHECK(cudaMemcpy(m->d_flags, flags, n, cudaMemcpyHostToDevice));
        BSX_CUDA_CHECK(cudaMemcpy(m->d_ins, insert, (size_t)n * 4, cudaMemcpyHostToDevice));
        BSX_CUDA_CHECK(cudaMemcpy(m->d_mate, mate_pos, (size_t)n * 4, cudaMemcpyHostToDevice));
        if (o->rm_dup) {
            rc = ensure_dup_table(m); if (rc) return rc;
            meth_claim_kernel<<<(n + 255) / 256, 256>>>(m->ix->d_seqinfo, m->ix->n_seq, m->d_first, *o, n, m->d_len, m->d_chr, m->d_pos, m->d_strand,
                                                       m->d_ins, m->d_mate, m->d_flags);
            BSX_CUDA_CHECK(cudaGetLastError());
        }
        const unsigned blocks = (unsigned)(((uint64_t)n * 32 + 255) / 256);
        const bool cyc = cycles_on(m);
        if (cyc) { rc = ensure_cycles(m); if (rc) return rc; }
        text_kernel(cyc, m->ct_snp != 0, m->d_conv != nullptr, m->d_pdr != nullptr, epi_on(m))<<<cyc ? std::min<unsigned>(blocks, (unsigned)m->resident[0]) : blocks, 256>>>(
            m->ix->d_refcat, m->ix->d_seqinfo, m->ix->n_seq, m->d_meth, m->d_depth, m->d_valid, o->rm_dup ? m->d_first : nullptr, *o, n, m->d_seq,
            m->stride, m->d_len, m->d_chr, m->d_pos, m->d_strand, m->d_ins, m->d_mate, m->d_flags, cyc ? mbias_args(m, 0) : MbiasArgs{}, m->d_confirm, m->d_snp,
            conv_args(m), pdr_args(m), epi_args(m));
        BSX_CUDA_CHECK(cudaGetLastError());
    }
    if (n_valid) {
        unsigned long long v = 0;
        BSX_CUDA_CHECK(cudaMemcpy(&v, m->d_valid, 8, cudaMemcpyDeviceToHost));
        *n_valid = v;
    }
    return BSX_OK;
}

// pile up the batch a mapper has just mapped (called by bsx_api.cu::run_slot on the batch's stream)
int bsx_meth_pile_mapped(bsx_meth *m, const bsx_meth_opts *o, int sam, int report_repeat_hits, uint32_t n, int mates, int readset, uint32_t stride,
                         const uint8_t *seq_a, const uint8_t *seq_b, const bsx_rec *out_a, const bsx_rec *out_b, const bsx_pair_rec *out_pair,
                         cudaStream_t st) {
    if (!m || !o || n == 0) return BSX_OK;
    if (m->combined) { bsx_set_error("bsx_meth: counters were already combined (-g); create a new bsx_meth"); return BSX_ERR_ARG; }
    m->started = true;
    const bool cyc = cycles_on(m);
    if (cyc) { int rc = ensure_cycles(m); if (rc) return rc; }
    if (o->rm_dup) {
        // file order = batch order: this batch's claims start when the previous batch has resolved its own (the batches
        // alternate between two streams).  Paired-end BSP output goes to two files, whose concatenation is the script's
        // order: that case is refused by bsx_mapper_attach_meth.
        int rc = ensure_dup_table(m); if (rc) return rc;
        BSX_CUDA_CHECK(cudaStreamWaitEvent(st, m->dup_order, 0));
        meth_claim_mapped_kernel<<<(unsigned)(((uint64_t)n * (uint64_t)mates + 255) / 256), 256, 0, st>>>(m->ix->d_seqinfo, m->ix->n_seq, m->d_first, *o, sam,
                                                                                                      report_repeat_hits, n, mates, out_a, out_b, out_pair);
        BSX_CUDA_CHECK(cudaGetLastError());
    }
    const unsigned blocks = (unsigned)(((uint64_t)n * (uint64_t)mates * 32 + 255) / 256);
    mapped_kernel(cyc, m->ct_snp != 0, m->d_conv != nullptr, m->d_pdr != nullptr, epi_on(m))<<<cyc ? std::min<unsigned>(blocks, (unsigned)m->resident[1]) : blocks, 256, 0, st>>>(
        m->ix->d_refcat, m->ix->d_seqinfo, m->ix->n_seq, m->d_meth, m->d_depth, m->d_valid, o->rm_dup ? m->d_first : nullptr, *o, sam,
        report_repeat_hits, n, mates, stride, seq_a, seq_b, out_a, out_b, out_pair, cyc ? mbias_args(m, readset) : MbiasArgs{}, m->d_confirm, m->d_snp,
        conv_args(m), pdr_args(m), epi_args(m));
    BSX_CUDA_CHECK(cudaGetLastError());
    if (o->rm_dup) BSX_CUDA_CHECK(cudaEventRecord(m->dup_order, st));
    return BSX_OK;
}

extern "C" int bsx_meth_valid_count(bsx_meth *m, uint64_t *n_valid) {
    if (!m || !n_valid) return BSX_ERR_ARG;
    BSX_CUDA_CHECK(cudaSetDevice(m->ix->device));
    BSX_CUDA_CHECK(cudaDeviceSynchronize());
    unsigned long long v = 0;
    BSX_CUDA_CHECK(cudaMemcpy(&v, m->d_valid, 8, cudaMemcpyDeviceToHost));
    *n_valid = v;
    return BSX_OK;
}

extern "C" int bsx_meth_download(bsx_meth *m, const bsx_meth_opts *o, uint32_t k, uint32_t *meth, uint32_t *depth) {
    if (!m || !o || k >= m->ix->n_seq) { bsx_set_error("bsx_meth_download: bad argument"); return BSX_ERR_ARG; }
    BSX_CUDA_CHECK(cudaSetDevice(m->ix->device));
    int rc = combine_once(m, o); if (rc) return rc;
    const size_t off = m->ix->anchor[k], cnt = m->ix->size[k];
    if (meth) BSX_CUDA_CHECK(cudaMemcpy(meth, m->d_meth + off, cnt * 4, cudaMemcpyDeviceToHost));
    if (depth) BSX_CUDA_CHECK(cudaMemcpy(depth, m->d_depth + off, cnt * 4, cudaMemcpyDeviceToHost));
    return BSX_OK;
}

extern "C" size_t bsx_meth_write(bsx_meth *m, const bsx_meth_opts *o, const char *const *seqs, const uint32_t *lens,
                                 const uint8_t *chroms, int threads, int fd, uint64_t *stats) {
    if (!m || !o || !seqs || !lens) { bsx_set_error("bsx_meth_write: bad argument"); return 0; }
    const bsx_index *ix = m->ix;
    threads = bsx_host_threads(threads);
    size_t written = 0;
    auto out = [&](const std::string &s) { size_t off = 0; while (off < s.size()) { ssize_t w = write(fd, s.data() + off, s.size() - off); if (w <= 0) return; off += (size_t)w; written += (size_t)w; } };
    const int snp_mode = m->ct_snp;
    out(snp_mode ? "chr\tpos\tstrand\tcontext\tratio\teff_CT_count\tC_count\tCT_count\trev_G_count\trev_GA_count\tCI_lower\tCI_upper\n"
                 : "chr\tpos\tstrand\tcontext\tratio\ttotal_C\tmethy_C\tCI_lower\tCI_upper\n");
    std::vector<uint32_t> order;
    for (uint32_t k = 0; k < ix->n_seq; k++) if (!chroms || chroms[k]) order.push_back(k);
    std::sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return ix->names[a] < ix->names[b]; });   // sorted(depth.keys())
    uint64_t nc = 0, nd = 0;
    const double z95 = 1.96, z95sq = 1.96 * 1.96;
    std::vector<uint32_t> hm, hd, hc, hs;
    for (uint32_t k : order) {
        const uint32_t L = ix->size[k];
        if (lens[k] != L) { bsx_set_error("bsx_meth_write: sequence %u has %u bases, the index %u", k, lens[k], L); return written; }
        hm.resize(L); hd.resize(L);
        if (bsx_meth_download(m, o, k, hm.data(), hd.data()) != BSX_OK) return written;
        if (snp_mode) { hc.resize(L); hs.resize(L); if (bsx_meth_download_ct_snp(m, o, k, hc.data(), hs.data()) != BSX_OK) return written; }
        const char *rs = seqs[k];
        const std::string &name = ix->names[k];
        std::vector<std::string> chunk((size_t)threads);
        std::vector<uint64_t> cnc((size_t)threads, 0), cnd((size_t)threads, 0);
        bsx_parallel(threads, L, [&](int t, size_t b, size_t e) {
            Sink s{&chunk[t]};
            uint64_t lc = 0, ld = 0;
            for (size_t i = b; i < e; i++) {
                const uint32_t d = hd[i];
                if ((long long)d < (long long)o->min_depth || d == 0) continue;
                lc++; ld += d;
                const uint32_t mm = hm[i];
                if (mm == 0 && !o->meth0) continue;
                // C/T SNP: the depth the ratio divides by; the line is dropped by `skip` at any SNP evidence and by
                // `correct` when no confirming evidence is left
                double eff = (double)d;
                uint64_t rg = 0, rga = 0;
                if (snp_mode) {
                    rg = hc[i]; rga = rg + hs[i];
                    if (snp_mode == BSX_CT_SNP_CORRECT) { if (rga) eff = (double)d * (double)rg / (double)rga; if (eff == 0) continue; }
                    else if (snp_mode == BSX_CT_SNP_SKIP && rg < rga) continue;
                }
                const double ratio = std::min((double)mm, eff) / eff;
                s.put(name.data(), name.size()); s.putc('\t'); s.putu(i + 1); s.putc('\t');
                const char rc = (char)(rs[i] >= 'a' && rs[i] <= 'z' ? rs[i] - 32 : rs[i]);
                s.putc(rc == 'C' ? '+' : '-'); s.putc('\t');
                // refcr[i-2:i+3] with Python's slice rules: for i < 2 the start counts from the sequence end, so a
                // sequence of 4 bases or fewer prints some of its last bases there, a longer one nothing
                const size_t c0 = i >= 2 ? i - 2 : (i + L >= 2 ? i + L - 2 : 0), c1 = std::min<size_t>(i + 3, L);
                for (size_t j = c0; j < c1; j++) s.putc((char)(rs[j] >= 'a' && rs[j] <= 'z' ? rs[j] - 32 : rs[j]));
                s.putc('\t'); s.putf3(ratio); s.putc('\t');
                if (snp_mode) { s.putf2(eff); s.putc('\t'); s.putu(mm); s.putc('\t'); s.putu(d); s.putc('\t'); s.putu(rg); s.putc('\t'); s.putu(rga); s.putc('\t'); }
                else { s.putu(d); s.putc('\t'); s.putu(mm); s.putc('\t'); }
                const double pmid = ratio + z95sq / (2 * eff);
                const double sd = z95 * pow(ratio * (1 - ratio) / eff + z95sq / (4 * eff * eff), 0.5);
                const double nm = 1 + z95sq / eff;
                s.putf3((pmid - sd) / nm); s.putc('\t'); s.putf3((pmid + sd) / nm); s.putc('\n');
            }
            cnc[t] = lc; cnd[t] = ld;
        });
        for (int t = 0; t < threads; t++) { out(chunk[t]); nc += cnc[t]; nd += cnd[t]; }
    }
    if (stats) { stats[0] = nc; stats[1] = nd; }
    return written;
}

extern "C" int bsx_meth_enable_ct_snp(bsx_meth *m, int mode) {
    if (!m) { bsx_set_error("bsx_meth_enable_ct_snp: bad argument"); return BSX_ERR_ARG; }
    if (m->started) { bsx_set_error("bsx_meth_enable_ct_snp: alignments were already piled up; enable C/T SNP evidence first"); return BSX_ERR_ARG; }
    if (mode != BSX_CT_SNP_NO_ACTION && mode != BSX_CT_SNP_CORRECT && mode != BSX_CT_SNP_SKIP) {
        bsx_set_error("bsx_meth_enable_ct_snp: mode must be BSX_CT_SNP_NO_ACTION, _CORRECT or _SKIP (got %d)", mode); return BSX_ERR_ARG; }
    if (!m->d_confirm) {
        BSX_CUDA_CHECK(cudaSetDevice(m->ix->device));
        const size_t bytes = m->ix->n_words * 16 * sizeof(uint32_t);
        if (cudaMalloc(&m->d_confirm, bytes) != cudaSuccess || cudaMalloc(&m->d_snp, bytes) != cudaSuccess) {
            cudaGetLastError(); cudaFree(m->d_confirm); cudaFree(m->d_snp); m->d_confirm = m->d_snp = nullptr;
            bsx_set_error("C/T SNP evidence: out of device memory (%zu bytes per evidence array, two arrays)", bytes); return BSX_ERR_CUDA; }
        BSX_CUDA_CHECK(cudaMemset(m->d_confirm, 0, bytes));
        BSX_CUDA_CHECK(cudaMemset(m->d_snp, 0, bytes));
    }
    m->ct_snp = mode;
    return BSX_OK;
}

int bsx_ct_snp_mode(const char *name) {
    return !strcmp(name, "no-action") ? BSX_CT_SNP_NO_ACTION : !strcmp(name, "correct") ? BSX_CT_SNP_CORRECT : !strcmp(name, "skip") ? BSX_CT_SNP_SKIP : 0;
}

extern "C" int bsx_meth_download_ct_snp(bsx_meth *m, const bsx_meth_opts *o, uint32_t k, uint32_t *confirm, uint32_t *snp) {
    if (!m || !o || k >= m->ix->n_seq) { bsx_set_error("bsx_meth_download_ct_snp: bad argument"); return BSX_ERR_ARG; }
    if (!m->ct_snp) { bsx_set_error("bsx_meth_download_ct_snp: C/T SNP evidence was not enabled (bsx_meth_enable_ct_snp)"); return BSX_ERR_ARG; }
    BSX_CUDA_CHECK(cudaSetDevice(m->ix->device));
    int rc = combine_once(m, o); if (rc) return rc;
    const size_t off = m->ix->anchor[k], cnt = m->ix->size[k];
    if (confirm) BSX_CUDA_CHECK(cudaMemcpy(confirm, m->d_confirm + off, cnt * 4, cudaMemcpyDeviceToHost));
    if (snp) BSX_CUDA_CHECK(cudaMemcpy(snp, m->d_snp + off, cnt * 4, cudaMemcpyDeviceToHost));
    return BSX_OK;
}

extern "C" int bsx_meth_enable_mbias(bsx_meth *m) {
    if (!m) { bsx_set_error("bsx_meth_enable_mbias: bad argument"); return BSX_ERR_ARG; }
    if (m->started) { bsx_set_error("bsx_meth_enable_mbias: alignments were already piled up; enable M-bias first"); return BSX_ERR_ARG; }
    m->mbias = true;
    return BSX_OK;
}

extern "C" int bsx_meth_set_ignore(bsx_meth *m, const int32_t ignore[4]) {
    if (!m || !ignore) { bsx_set_error("bsx_meth_set_ignore: bad argument"); return BSX_ERR_ARG; }
    if (m->started) { bsx_set_error("bsx_meth_set_ignore: alignments were already piled up; set the exclusion first"); return BSX_ERR_ARG; }
    for (int i = 0; i < 4; i++)
        if (ignore[i] < 0) { bsx_set_error("bsx_meth_set_ignore: cycle counts must be >= 0 (got %d)", ignore[i]); return BSX_ERR_ARG; }
    for (int i = 0; i < 4; i++) m->ignore[i] = ignore[i];
    return BSX_OK;
}

extern "C" int bsx_meth_mbias(bsx_meth *m, uint64_t *out, uint64_t *overflow) {
    if (!m || !out) { bsx_set_error("bsx_meth_mbias: bad argument"); return BSX_ERR_ARG; }
    if (!m->mbias) { bsx_set_error("bsx_meth_mbias: M-bias was not enabled (bsx_meth_enable_mbias)"); return BSX_ERR_ARG; }
    BSX_CUDA_CHECK(cudaSetDevice(m->ix->device));
    BSX_CUDA_CHECK(cudaDeviceSynchronize());           // in-process batches flush from two streams
    std::vector<unsigned long long> h(MBIAS_BINS + 1, 0ull);
    if (m->d_mbias) BSX_CUDA_CHECK(cudaMemcpy(h.data(), m->d_mbias, h.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    for (int b = 0; b < MBIAS_BINS; b++) out[b] = h[b];
    if (overflow) *overflow = h[MBIAS_BINS];
    return BSX_OK;
}

// the report to fd; *overflow (may be NULL) from the same download
static size_t write_mbias(bsx_meth *m, int fd, uint64_t *overflow) {
    std::vector<uint64_t> h(MBIAS_BINS);
    if (bsx_meth_mbias(m, h.data(), overflow) != BSX_OK) return 0;
    std::string s = "context\tread\tcycle\tmethylated\tunmethylated\tratio\n";
    Sink o{&s};
    static const char *const ctx[3] = {"CpG", "CHG", "CHH"};
    for (int c = 0; c < 3; c++)
        for (int r = 0; r < 2; r++)
            for (int y = 0; y < BSX_MBIAS_CYCLES; y++) {
                const uint64_t *b = &h[((size_t)(r * 3 + c) * BSX_MBIAS_CYCLES + y) * 2];
                if (b[0] + b[1] == 0) continue;
                o.put(ctx[c], 3); o.putc('\t'); o.putc((char)('1' + r)); o.putc('\t'); o.putu((unsigned long long)y + 1); o.putc('\t');
                o.putu(b[0]); o.putc('\t'); o.putu(b[1]); o.putc('\t'); o.putf3((double)b[0] / (double)(b[0] + b[1])); o.putc('\n');
            }
    size_t off = 0;
    while (off < s.size()) { const ssize_t w = write(fd, s.data() + off, s.size() - off); if (w <= 0) break; off += (size_t)w; }
    return off;
}

extern "C" size_t bsx_meth_write_mbias(bsx_meth *m, int fd) { return write_mbias(m, fd, nullptr); }

int bsx_meth_write_mbias_file(bsx_meth *m, const char *path) {
    const int fd = open(path, O_WRONLY | O_CREAT | O_TRUNC, 0644);
    if (fd < 0) { fprintf(stderr, "failed to open M-bias output file: %s\n", path); return BSX_ERR_IO; }
    uint64_t over = 0;
    const size_t w = write_mbias(m, fd, &over);
    close(fd);
    if (w == 0) { fprintf(stderr, "%s\n", bsx_last_error()); return BSX_ERR_IO; }
    if (over) fprintf(stderr, "warning: %llu methylation calls at cycle %d or later are in the table but not in the M-bias report\n",
                      (unsigned long long)over, BSX_MBIAS_CYCLES + 1);
    return BSX_OK;
}

extern "C" int bsx_meth_enable_conversion_filter(bsx_meth *m, int32_t threshold) {
    if (!m) { bsx_set_error("bsx_meth_enable_conversion_filter: bad argument"); return BSX_ERR_ARG; }
    if (m->started) { bsx_set_error("bsx_meth_enable_conversion_filter: alignments were already piled up; enable the conversion filter first"); return BSX_ERR_ARG; }
    if (threshold < 0 || threshold > BSX_CONV_BINS - 1) {
        bsx_set_error("bsx_meth_enable_conversion_filter: threshold must be 0..%d (got %d)", BSX_CONV_BINS - 1, (int)threshold); return BSX_ERR_ARG; }
    if (!m->d_conv) {
        BSX_CUDA_CHECK(cudaSetDevice(m->ix->device));
        BSX_CUDA_CHECK(cudaMalloc(&m->d_conv, BSX_CONV_BINS * sizeof(unsigned long long)));
        BSX_CUDA_CHECK(cudaMemset(m->d_conv, 0, BSX_CONV_BINS * sizeof(unsigned long long)));
    }
    m->conv_threshold = threshold;
    return BSX_OK;
}

extern "C" int bsx_meth_conversion(bsx_meth *m, uint64_t *out, uint64_t *dropped) {
    if (!m || !out) { bsx_set_error("bsx_meth_conversion: bad argument"); return BSX_ERR_ARG; }
    if (!m->d_conv) { bsx_set_error("bsx_meth_conversion: the conversion filter was not enabled (bsx_meth_enable_conversion_filter)"); return BSX_ERR_ARG; }
    BSX_CUDA_CHECK(cudaSetDevice(m->ix->device));
    BSX_CUDA_CHECK(cudaDeviceSynchronize());           // in-process batches flush from two streams
    unsigned long long h[BSX_CONV_BINS];
    BSX_CUDA_CHECK(cudaMemcpy(h, m->d_conv, sizeof h, cudaMemcpyDeviceToHost));
    uint64_t d = 0;
    for (int b = 0; b < BSX_CONV_BINS; b++) { out[b] = h[b]; if (m->conv_threshold && b >= m->conv_threshold) d += h[b]; }
    if (dropped) *dropped = d;
    return BSX_OK;
}

extern "C" size_t bsx_meth_write_conversion(bsx_meth *m, int fd) {
    uint64_t h[BSX_CONV_BINS];
    if (bsx_meth_conversion(m, h, nullptr) != BSX_OK) return 0;
    std::string s = "methylated_nonCpG_calls\talignments\tdropped\n";
    Sink o{&s};
    for (int b = 0; b < BSX_CONV_BINS; b++) {
        if (!h[b]) continue;
        o.putu((unsigned long long)b);
        if (b == BSX_CONV_BINS - 1) o.putc('+');
        o.putc('\t'); o.putu(h[b]); o.putc('\t'); o.putc(m->conv_threshold && b >= m->conv_threshold ? '1' : '0'); o.putc('\n');
    }
    size_t off = 0;
    while (off < s.size()) { const ssize_t w = write(fd, s.data() + off, s.size() - off); if (w <= 0) return 0; off += (size_t)w; }
    return off;
}

int bsx_meth_write_conversion_file(bsx_meth *m, const char *path) {
    if (path) {
        const int fd = open(path, O_WRONLY | O_CREAT | O_TRUNC, 0644);
        if (fd < 0) { fprintf(stderr, "failed to open conversion report file: %s\n", path); return BSX_ERR_IO; }
        const size_t w = bsx_meth_write_conversion(m, fd);
        close(fd);
        if (w == 0) { fprintf(stderr, "%s\n", bsx_last_error()); return BSX_ERR_IO; }
    }
    uint64_t h[BSX_CONV_BINS], dropped = 0, valid = 0;
    if (bsx_meth_conversion(m, h, &dropped) != BSX_OK || bsx_meth_valid_count(m, &valid) != BSX_OK) { fprintf(stderr, "%s\n", bsx_last_error()); return BSX_ERR_CUDA; }
    if (m->conv_threshold)
        fprintf(stderr, "conversion filter: %llu of %llu valid mappings dropped (>= %d methylated non-CpG calls)\n", (unsigned long long)dropped,
                (unsigned long long)valid, m->conv_threshold);
    else fprintf(stderr, "conversion filter: 0 of %llu valid mappings dropped (report only)\n", (unsigned long long)valid);
    return BSX_OK;
}

extern "C" int bsx_meth_enable_pdr(bsx_meth *m, int32_t min_cpg) {
    if (!m) { bsx_set_error("bsx_meth_enable_pdr: bad argument"); return BSX_ERR_ARG; }
    if (m->started) { bsx_set_error("bsx_meth_enable_pdr: alignments were already piled up; enable PDR first"); return BSX_ERR_ARG; }
    if (min_cpg < 1 || min_cpg > 255) { bsx_set_error("bsx_meth_enable_pdr: the minimum of CpG calls must be 1..255 (got %d)", (int)min_cpg); return BSX_ERR_ARG; }
    if (!m->d_pdr) {
        BSX_CUDA_CHECK(cudaSetDevice(m->ix->device));
        const size_t bytes = m->ix->n_words * 16 * sizeof(uint32_t);
        if (cudaMalloc(&m->d_conc, bytes) != cudaSuccess || cudaMalloc(&m->d_disc, bytes) != cudaSuccess ||
            cudaMalloc(&m->d_pdr, 2 * sizeof(unsigned long long)) != cudaSuccess) {
            cudaGetLastError(); cudaFree(m->d_conc); cudaFree(m->d_disc); cudaFree(m->d_pdr); m->d_conc = m->d_disc = nullptr; m->d_pdr = nullptr;
            bsx_set_error("PDR: out of device memory (%zu bytes per concordance array, two arrays)", bytes); return BSX_ERR_CUDA; }
        BSX_CUDA_CHECK(cudaMemset(m->d_conc, 0, bytes));
        BSX_CUDA_CHECK(cudaMemset(m->d_disc, 0, bytes));
        BSX_CUDA_CHECK(cudaMemset(m->d_pdr, 0, 2 * sizeof(unsigned long long)));
    }
    m->pdr_min_cpg = (uint32_t)min_cpg;
    return BSX_OK;
}

extern "C" int bsx_meth_download_pdr(bsx_meth *m, const bsx_meth_opts *o, uint32_t k, uint32_t *concordant, uint32_t *discordant) {
    if (!m || !o || k >= m->ix->n_seq) { bsx_set_error("bsx_meth_download_pdr: bad argument"); return BSX_ERR_ARG; }
    if (!m->d_pdr) { bsx_set_error("bsx_meth_download_pdr: PDR was not enabled (bsx_meth_enable_pdr)"); return BSX_ERR_ARG; }
    BSX_CUDA_CHECK(cudaSetDevice(m->ix->device));
    int rc = combine_once(m, o); if (rc) return rc;
    const size_t off = m->ix->anchor[k], cnt = m->ix->size[k];
    if (concordant) BSX_CUDA_CHECK(cudaMemcpy(concordant, m->d_conc + off, cnt * 4, cudaMemcpyDeviceToHost));
    if (discordant) BSX_CUDA_CHECK(cudaMemcpy(discordant, m->d_disc + off, cnt * 4, cudaMemcpyDeviceToHost));
    return BSX_OK;
}

extern "C" int bsx_meth_pdr(bsx_meth *m, uint64_t *informative, uint64_t *discordant) {
    if (!m) { bsx_set_error("bsx_meth_pdr: bad argument"); return BSX_ERR_ARG; }
    if (!m->d_pdr) { bsx_set_error("bsx_meth_pdr: PDR was not enabled (bsx_meth_enable_pdr)"); return BSX_ERR_ARG; }
    BSX_CUDA_CHECK(cudaSetDevice(m->ix->device));
    BSX_CUDA_CHECK(cudaDeviceSynchronize());           // in-process batches flush from two streams
    unsigned long long h[2];
    BSX_CUDA_CHECK(cudaMemcpy(h, m->d_pdr, sizeof h, cudaMemcpyDeviceToHost));
    if (informative) *informative = h[0];
    if (discordant) *discordant = h[1];
    return BSX_OK;
}

extern "C" size_t bsx_meth_write_pdr(bsx_meth *m, const bsx_meth_opts *o, const char *const *seqs, const uint32_t *lens, const uint8_t *chroms,
                                     int threads, int fd) {
    if (!m || !o || !seqs || !lens) { bsx_set_error("bsx_meth_write_pdr: bad argument"); return 0; }
    if (!m->d_pdr) { bsx_set_error("bsx_meth_write_pdr: PDR was not enabled (bsx_meth_enable_pdr)"); return 0; }
    const bsx_index *ix = m->ix;
    threads = bsx_host_threads(threads);
    size_t written = 0;
    auto out = [&](const std::string &s) {
        size_t off = 0;
        while (off < s.size()) { const ssize_t w = write(fd, s.data() + off, s.size() - off); if (w <= 0) return false; off += (size_t)w; written += (size_t)w; }
        return true;
    };
    if (!out("chr\tpos\tstrand\tconcordant\tdiscordant\tPDR\n")) return 0;
    std::vector<uint32_t> order;
    for (uint32_t k = 0; k < ix->n_seq; k++) if (!chroms || chroms[k]) order.push_back(k);
    std::sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return ix->names[a] < ix->names[b]; });   // the table's order
    const int snp_mode = m->ct_snp == BSX_CT_SNP_SKIP || m->ct_snp == BSX_CT_SNP_CORRECT ? m->ct_snp : 0;
    const uint64_t min_n = (uint64_t)std::max(o->min_depth, 1);
    std::vector<uint32_t> hc, hd, ec, es;
    for (uint32_t k : order) {
        const uint32_t L = ix->size[k];
        if (lens[k] != L) { bsx_set_error("bsx_meth_write_pdr: sequence %u has %u bases, the index %u", k, lens[k], L); return 0; }
        hc.resize(L); hd.resize(L);
        if (bsx_meth_download_pdr(m, o, k, hc.data(), hd.data()) != BSX_OK) return 0;
        if (snp_mode) { ec.resize(L); es.resize(L); if (bsx_meth_download_ct_snp(m, o, k, ec.data(), es.data()) != BSX_OK) return 0; }
        const char *rs = seqs[k];
        const std::string &name = ix->names[k];
        std::vector<std::string> chunk((size_t)threads);
        bsx_parallel(threads, L, [&](int t, size_t b, size_t e) {
            Sink s{&chunk[t]};
            for (size_t i = b; i < e; i++) {
                const uint64_t c = hc[i], d = hd[i];
                if (c + d < min_n) continue;
                // the C/T SNP mode drops the line as it drops the table's: `skip` at any SNP evidence, `correct` when eff == 0
                if (snp_mode == BSX_CT_SNP_SKIP && es[i]) continue;
                if (snp_mode == BSX_CT_SNP_CORRECT && es[i] && !ec[i]) continue;
                s.put(name.data(), name.size()); s.putc('\t'); s.putu(i + 1); s.putc('\t');
                const char rc = (char)(rs[i] >= 'a' && rs[i] <= 'z' ? rs[i] - 32 : rs[i]);
                s.putc(rc == 'C' ? '+' : '-'); s.putc('\t');
                s.putu(c); s.putc('\t'); s.putu(d); s.putc('\t'); s.putf3((double)d / (double)(c + d)); s.putc('\n');
            }
        });
        for (int t = 0; t < threads; t++) if (!out(chunk[t])) return 0;
    }
    return written;
}

int bsx_meth_write_pdr_file(bsx_meth *m, const bsx_meth_opts *o, const char *const *seqs, const uint32_t *lens, const uint8_t *chroms, int threads,
                            const char *path) {
    const int fd = open(path, O_WRONLY | O_CREAT | O_TRUNC, 0644);
    if (fd < 0) { fprintf(stderr, "failed to open PDR output file: %s\n", path); return BSX_ERR_IO; }
    const size_t w = bsx_meth_write_pdr(m, o, seqs, lens, chroms, threads, fd);
    close(fd);
    if (w == 0) { fprintf(stderr, "%s\n", bsx_last_error()); return BSX_ERR_IO; }
    uint64_t inf = 0, disc = 0, valid = 0;
    if (bsx_meth_pdr(m, &inf, &disc) != BSX_OK || bsx_meth_valid_count(m, &valid) != BSX_OK) { fprintf(stderr, "%s\n", bsx_last_error()); return BSX_ERR_CUDA; }
    fprintf(stderr, "PDR: %llu of %llu valid mappings informative (>= %u CpG calls), %llu discordant\n", (unsigned long long)inf, (unsigned long long)valid,
            m->pdr_min_cpg, (unsigned long long)disc);
    return BSX_OK;
}

extern "C" int bsx_meth_enable_epialleles(bsx_meth *m) {
    if (!m) { bsx_set_error("bsx_meth_enable_epialleles: bad argument"); return BSX_ERR_ARG; }
    if (m->started) { bsx_set_error("bsx_meth_enable_epialleles: alignments were already piled up; enable epialleles first"); return BSX_ERR_ARG; }
    if (m->d_epi) { bsx_set_error("bsx_meth_enable_epialleles: epialleles are already enabled"); return BSX_ERR_ARG; }
    BSX_CUDA_CHECK(cudaSetDevice(m->ix->device));
    const int rc = ensure_cpg_rank(m, "epialleles");
    if (rc) return rc;
    const uint64_t sites = m->cpg_sites;
    auto undo = [m]() { cudaFree(m->d_epi); cudaFree(m->d_epi_count); m->d_epi = nullptr; m->d_epi_count = nullptr; };
    const size_t bytes = (size_t)std::max<uint64_t>(sites, 1u) * 16 * sizeof(uint32_t);
    if (cudaMalloc(&m->d_epi, bytes) != cudaSuccess || cudaMalloc(&m->d_epi_count, 2 * sizeof(unsigned long long)) != cudaSuccess) {
        cudaGetLastError(); undo();
        bsx_set_error("epialleles: out of device memory (%zu bytes for the pattern counters of %llu CpG sites)", bytes, (unsigned long long)sites); return BSX_ERR_CUDA; }
    if (cudaMemset(m->d_epi, 0, bytes) != cudaSuccess || cudaMemset(m->d_epi_count, 0, 2 * sizeof(unsigned long long)) != cudaSuccess) {
        cudaGetLastError(); undo(); bsx_set_error("epialleles: cudaMemset failed"); return BSX_ERR_CUDA; }
    return BSX_OK;
}

// the CpG sites of sequence k: their positions in the sequence (may be NULL), their number and the rank of the first,
// from the device's packed reference and rank index (the rule of cpg_rank, so that the ranks line up)
static int epi_sites(bsx_meth *m, uint32_t k, std::vector<uint32_t> *pos, uint64_t *n, uint64_t *rank0) {
    const bsx_index *ix = m->ix;
    const uint64_t a0 = ix->anchor[k], L = ix->size[k];
    const uint64_t w0 = a0 >> 4, w1 = std::min<uint64_t>((a0 + L) >> 4, ix->n_words - 1);   // the words holding [a0, a0 + L], and the next
    std::vector<uint32_t> w((size_t)(w1 - w0 + 2), 0u);
    BSX_CUDA_CHECK(cudaMemcpy(w.data(), ix->d_refcat + w0, (size_t)(w1 - w0 + 1) * 4, cudaMemcpyDeviceToHost));
    uint32_t r = 0;
    BSX_CUDA_CHECK(cudaMemcpy(&r, m->d_cpg_rank + w0, 4, cudaMemcpyDeviceToHost));
    const uint32_t lead = (uint32_t)(a0 & 15);
    r += (uint32_t)__builtin_popcount(cpg_mask(w[0], 0u) & ~(0xffffffffu >> (2 * lead)));
    uint64_t cnt = 0;
    for (uint64_t q = a0 - (a0 & 15); q < a0 + L; q += 16) {
        const size_t wi = (size_t)((q >> 4) - w0);
        uint32_t s = cpg_mask(w[wi], w[wi + 1]);
        while (s) {
            const int b = 31 - __builtin_clz(s);
            s &= ~(1u << b);
            const uint64_t c = q + (uint64_t)((30 - b) >> 1);
            if (c < a0 || c >= a0 + L) continue;
            if (pos) pos->push_back((uint32_t)(c - a0));
            cnt++;
        }
    }
    *n = cnt; *rank0 = r;
    return BSX_OK;
}

extern "C" int bsx_meth_cpg_sites(bsx_meth *m, uint32_t k, uint64_t *n) {
    if (!m || !n || k >= m->ix->n_seq) { bsx_set_error("bsx_meth_cpg_sites: bad argument"); return BSX_ERR_ARG; }
    if (!m->d_cpg_rank) { bsx_set_error("bsx_meth_cpg_sites: epialleles or MHL were not enabled (bsx_meth_enable_epialleles, bsx_meth_enable_mhl)"); return BSX_ERR_ARG; }
    BSX_CUDA_CHECK(cudaSetDevice(m->ix->device));
    uint64_t r0 = 0;
    return epi_sites(m, k, nullptr, n, &r0);
}

extern "C" int bsx_meth_download_epialleles(bsx_meth *m, uint32_t k, uint32_t *site_pos, uint32_t *counts) {
    if (!m || k >= m->ix->n_seq) { bsx_set_error("bsx_meth_download_epialleles: bad argument"); return BSX_ERR_ARG; }
    if (!m->d_epi) { bsx_set_error("bsx_meth_download_epialleles: epialleles were not enabled (bsx_meth_enable_epialleles)"); return BSX_ERR_ARG; }
    BSX_CUDA_CHECK(cudaSetDevice(m->ix->device));
    BSX_CUDA_CHECK(cudaDeviceSynchronize());           // in-process batches pile up from two streams
    std::vector<uint32_t> pos;
    uint64_t n = 0, r0 = 0;
    int rc = epi_sites(m, k, &pos, &n, &r0); if (rc) return rc;
    if (site_pos && n) memcpy(site_pos, pos.data(), n * 4);
    if (counts && n) BSX_CUDA_CHECK(cudaMemcpy(counts, m->d_epi + r0 * 16, n * 16 * 4, cudaMemcpyDeviceToHost));
    return BSX_OK;
}

extern "C" int bsx_meth_epialleles(bsx_meth *m, uint64_t *spanning, uint64_t *windows) {
    if (!m) { bsx_set_error("bsx_meth_epialleles: bad argument"); return BSX_ERR_ARG; }
    if (!m->d_epi) { bsx_set_error("bsx_meth_epialleles: epialleles were not enabled (bsx_meth_enable_epialleles)"); return BSX_ERR_ARG; }
    BSX_CUDA_CHECK(cudaSetDevice(m->ix->device));
    BSX_CUDA_CHECK(cudaDeviceSynchronize());           // in-process batches flush from two streams
    unsigned long long h[2];
    BSX_CUDA_CHECK(cudaMemcpy(h, m->d_epi_count, sizeof h, cudaMemcpyDeviceToHost));
    if (spanning) *spanning = h[0];
    if (windows) *windows = h[1];
    return BSX_OK;
}

extern "C" size_t bsx_meth_write_epialleles(bsx_meth *m, const bsx_meth_opts *o, const char *const *seqs, const uint32_t *lens, const uint8_t *chroms,
                                            int threads, int fd) {
    if (!m || !o || !seqs || !lens) { bsx_set_error("bsx_meth_write_epialleles: bad argument"); return 0; }
    if (!m->d_epi) { bsx_set_error("bsx_meth_write_epialleles: epialleles were not enabled (bsx_meth_enable_epialleles)"); return 0; }
    const bsx_index *ix = m->ix;
    if (cudaSetDevice(ix->device) != cudaSuccess || cudaDeviceSynchronize() != cudaSuccess) {   // in-process batches pile up from two streams
        bsx_set_error("bsx_meth_write_epialleles: %s", cudaGetErrorString(cudaGetLastError())); return 0; }
    threads = bsx_host_threads(threads);
    size_t written = 0;
    auto out = [&](const std::string &s) {
        size_t off = 0;
        while (off < s.size()) { const ssize_t w = write(fd, s.data() + off, s.size() - off); if (w <= 0) return false; off += (size_t)w; written += (size_t)w; }
        return true;
    };
    if (!out("chr\tstart\tend\treads\tlevel\tentropy\tEPM\tpatterns\n")) return 0;
    std::vector<uint32_t> order;
    for (uint32_t k = 0; k < ix->n_seq; k++) if (!chroms || chroms[k]) order.push_back(k);
    std::sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return ix->names[a] < ix->names[b]; });   // the table's order
    // `correct` cannot rescale a pattern, so both SNP modes drop a window with SNP evidence at any of its eight bases
    const bool snp_drop = m->ct_snp == BSX_CT_SNP_SKIP || m->ct_snp == BSX_CT_SNP_CORRECT;
    const uint64_t min_n = (uint64_t)std::max(o->min_depth, 1);
    std::vector<uint32_t> pos, cnt, ec, es;
    for (uint32_t k : order) {
        const uint32_t L = ix->size[k];
        if (lens[k] != L) { bsx_set_error("bsx_meth_write_epialleles: sequence %u has %u bases, the index %u", k, lens[k], L); return 0; }
        uint64_t n = 0, r0 = 0;
        pos.clear();
        if (epi_sites(m, k, &pos, &n, &r0) != BSX_OK) return 0;
        if (n < BSX_EPI_CPGS) continue;
        cnt.resize(n * 16);
        if (cudaMemcpy(cnt.data(), m->d_epi + r0 * 16, n * 16 * 4, cudaMemcpyDeviceToHost) != cudaSuccess) {
            bsx_set_error("bsx_meth_write_epialleles: counter download failed: %s", cudaGetErrorString(cudaGetLastError())); return 0; }
        if (snp_drop) { ec.resize(L); es.resize(L); if (bsx_meth_download_ct_snp(m, o, k, ec.data(), es.data()) != BSX_OK) return 0; }
        const std::string &name = ix->names[k];
        std::vector<std::string> chunk((size_t)threads);
        bsx_parallel(threads, (size_t)(n - (BSX_EPI_CPGS - 1)), [&](int t, size_t b, size_t e) {
            Sink s{&chunk[t]};
            for (size_t j = b; j < e; j++) {
                const uint32_t *c = &cnt[j * 16];
                uint64_t reads = 0, meth = 0;
                for (int i = 0; i < 16; i++) { reads += c[i]; meth += (uint64_t)c[i] * (uint64_t)__builtin_popcount((unsigned)i); }
                if (reads < min_n) continue;
                if (snp_drop) {
                    bool ev = false;
                    for (int t4 = 0; t4 < BSX_EPI_CPGS; t4++) ev = ev || es[pos[j + t4]] || es[pos[j + t4] + 1];
                    if (ev) continue;
                }
                // ascending i in double, as the oracle sums them
                double h = 0.0, sq = 0.0;
                for (int i = 0; i < 16; i++) {
                    if (!c[i]) continue;
                    const double p = (double)c[i] / (double)reads;
                    h += p * log2(p); sq += p * p;
                }
                s.put(name.data(), name.size()); s.putc('\t'); s.putu(pos[j] + 1ull); s.putc('\t'); s.putu(pos[j + BSX_EPI_CPGS - 1] + 2ull); s.putc('\t');
                s.putu(reads); s.putc('\t'); s.putf4((double)meth / (double)(4 * reads)); s.putc('\t'); s.putf4((0.0 - h) / 4.0); s.putc('\t');
                s.putf4(1.0 - sq); s.putc('\t');
                for (int i = 0; i < 16; i++) { if (i) s.putc(','); s.putu(c[i]); }
                s.putc('\n');
            }
        });
        for (int t = 0; t < threads; t++) if (!out(chunk[t])) return 0;
    }
    return written;
}

int bsx_meth_write_epialleles_file(bsx_meth *m, const bsx_meth_opts *o, const char *const *seqs, const uint32_t *lens, const uint8_t *chroms, int threads,
                                   const char *path) {
    const int fd = open(path, O_WRONLY | O_CREAT | O_TRUNC, 0644);
    if (fd < 0) { fprintf(stderr, "failed to open epiallele output file: %s\n", path); return BSX_ERR_IO; }
    const size_t w = bsx_meth_write_epialleles(m, o, seqs, lens, chroms, threads, fd);
    close(fd);
    if (w == 0) { fprintf(stderr, "%s\n", bsx_last_error()); return BSX_ERR_IO; }
    uint64_t spanning = 0, windows = 0, valid = 0;
    if (bsx_meth_epialleles(m, &spanning, &windows) != BSX_OK || bsx_meth_valid_count(m, &valid) != BSX_OK) { fprintf(stderr, "%s\n", bsx_last_error()); return BSX_ERR_CUDA; }
    fprintf(stderr, "epialleles: %llu of %llu valid mappings span a %d-CpG window, %llu window patterns counted\n", (unsigned long long)spanning,
            (unsigned long long)valid, BSX_EPI_CPGS, (unsigned long long)windows);
    return BSX_OK;
}

extern "C" int bsx_meth_enable_mhl(bsx_meth *m) {
    if (!m) { bsx_set_error("bsx_meth_enable_mhl: bad argument"); return BSX_ERR_ARG; }
    if (m->started) { bsx_set_error("bsx_meth_enable_mhl: alignments were already piled up; enable MHL first"); return BSX_ERR_ARG; }
    if (m->d_mhl) { bsx_set_error("bsx_meth_enable_mhl: MHL is already enabled"); return BSX_ERR_ARG; }
    BSX_CUDA_CHECK(cudaSetDevice(m->ix->device));
    const int rc = ensure_cpg_rank(m, "MHL");
    if (rc) return rc;
    auto undo = [m]() { cudaFree(m->d_mhl); cudaFree(m->d_mhl_count); m->d_mhl = nullptr; m->d_mhl_count = nullptr; };
    const size_t bytes = (size_t)std::max<uint64_t>(m->cpg_sites, 1u) * 3 * BSX_MHL_MAX_LEN * sizeof(uint32_t);
    if (cudaMalloc(&m->d_mhl, bytes) != cudaSuccess || cudaMalloc(&m->d_mhl_count, 2 * sizeof(unsigned long long)) != cudaSuccess) {
        cudaGetLastError(); undo();
        bsx_set_error("MHL: out of device memory (%zu bytes for the run counters of %llu CpG sites)", bytes, (unsigned long long)m->cpg_sites); return BSX_ERR_CUDA; }
    if (cudaMemset(m->d_mhl, 0, bytes) != cudaSuccess || cudaMemset(m->d_mhl_count, 0, 2 * sizeof(unsigned long long)) != cudaSuccess) {
        cudaGetLastError(); undo(); bsx_set_error("MHL: cudaMemset failed"); return BSX_ERR_CUDA; }
    return BSX_OK;
}

extern "C" int bsx_meth_download_mhl(bsx_meth *m, uint32_t k, uint32_t *site_pos, uint32_t *counts) {
    if (!m || k >= m->ix->n_seq) { bsx_set_error("bsx_meth_download_mhl: bad argument"); return BSX_ERR_ARG; }
    if (!m->d_mhl) { bsx_set_error("bsx_meth_download_mhl: MHL was not enabled (bsx_meth_enable_mhl)"); return BSX_ERR_ARG; }
    BSX_CUDA_CHECK(cudaSetDevice(m->ix->device));
    BSX_CUDA_CHECK(cudaDeviceSynchronize());           // in-process batches pile up from two streams
    std::vector<uint32_t> pos;
    uint64_t n = 0, r0 = 0;
    int rc = epi_sites(m, k, &pos, &n, &r0); if (rc) return rc;
    if (site_pos && n) memcpy(site_pos, pos.data(), n * 4);
    if (counts && n) BSX_CUDA_CHECK(cudaMemcpy(counts, m->d_mhl + r0 * 3 * BSX_MHL_MAX_LEN, n * 3 * BSX_MHL_MAX_LEN * 4, cudaMemcpyDeviceToHost));
    return BSX_OK;
}

extern "C" int bsx_meth_mhl(bsx_meth *m, uint64_t *alignments, uint64_t *calls) {
    if (!m) { bsx_set_error("bsx_meth_mhl: bad argument"); return BSX_ERR_ARG; }
    if (!m->d_mhl) { bsx_set_error("bsx_meth_mhl: MHL was not enabled (bsx_meth_enable_mhl)"); return BSX_ERR_ARG; }
    BSX_CUDA_CHECK(cudaSetDevice(m->ix->device));
    BSX_CUDA_CHECK(cudaDeviceSynchronize());           // in-process batches flush from two streams
    unsigned long long h[2];
    BSX_CUDA_CHECK(cudaMemcpy(h, m->d_mhl_count, sizeof h, cudaMemcpyDeviceToHost));
    if (alignments) *alignments = h[0];
    if (calls) *calls = h[1];
    return BSX_OK;
}

extern "C" int bsx_meth_regions_mhl(bsx_meth *m, const bsx_meth_opts *o, uint64_t n, const uint32_t *seq, const uint64_t *start, const uint64_t *end,
                                    uint64_t *sites, uint64_t *out) {
    if (!m || !o || (n && (!seq || !start || !end || !sites || !out))) { bsx_set_error("bsx_meth_regions_mhl: bad argument"); return BSX_ERR_ARG; }
    if (!m->d_mhl) { bsx_set_error("bsx_meth_regions_mhl: MHL was not enabled (bsx_meth_enable_mhl)"); return BSX_ERR_ARG; }
    const bsx_index *ix = m->ix;
    for (uint64_t r = 0; r < n; r++) {
        if (seq[r] >= ix->n_seq) { bsx_set_error("bsx_meth_regions_mhl: region %llu: sequence %u of %u", (unsigned long long)r, seq[r], ix->n_seq); return BSX_ERR_ARG; }
        if (start[r] > end[r]) { bsx_set_error("bsx_meth_regions_mhl: region %llu: start %llu > end %llu", (unsigned long long)r, (unsigned long long)start[r],
                                               (unsigned long long)end[r]); return BSX_ERR_ARG; }
    }
    BSX_CUDA_CHECK(cudaSetDevice(ix->device));
    BSX_CUDA_CHECK(cudaDeviceSynchronize());           // in-process batches pile up on the mapper's streams
    if (n == 0) return BSX_OK;
    const uint64_t cap = std::min<uint64_t>(n, MHL_SLICE);
    const bool cuts = m->ct_snp == BSX_CT_SNP_SKIP || m->ct_snp == BSX_CT_SNP_CORRECT;
    const size_t cut_words = (size_t)((m->cpg_sites + 31) / 32) + 1;
    uint32_t *d_chunks = nullptr, *d_cut = nullptr; uint2 *d_pos = nullptr, *d_span = nullptr; unsigned long long *d_out = nullptr;
    if (cudaMalloc(&d_chunks, (cap + 1) * 4) != cudaSuccess || cudaMalloc(&d_pos, cap * 8) != cudaSuccess || cudaMalloc(&d_span, cap * 8) != cudaSuccess ||
        cudaMalloc(&d_out, cap * 48 * 8) != cudaSuccess || (cuts && cudaMalloc(&d_cut, cut_words * 4) != cudaSuccess)) {
        cudaGetLastError(); cudaFree(d_chunks); cudaFree(d_pos); cudaFree(d_span); cudaFree(d_out); cudaFree(d_cut);
        bsx_set_error("bsx_meth_regions_mhl: out of device memory"); return BSX_ERR_CUDA; }
    auto run = [&]() -> int {
        if (cuts) {
            BSX_CUDA_CHECK(cudaMemset(d_cut, 0, cut_words * 4));
            mhl_cut_kernel<<<(unsigned)((ix->n_words + 255) / 256), 256>>>(ix->d_refcat, ix->n_words, m->d_cpg_rank, m->d_snp, d_cut);
            BSX_CUDA_CHECK(cudaGetLastError());
        }
        int dev = 0, sms = 0, per_sm = 0;
        BSX_CUDA_CHECK(cudaGetDevice(&dev));
        BSX_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        BSX_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, meth_mhl_region_kernel, 256, 0));
        std::vector<uint2> pos, span;
        for (uint64_t r0 = 0; r0 < n; r0 += cap) {
            const uint32_t k = (uint32_t)std::min(cap, n - r0);
            pos.resize(k); span.resize(k);
            for (uint32_t i = 0; i < k; i++) {
                const uint32_t sq = seq[r0 + i], len = ix->size[sq];
                const uint64_t lo = std::min<uint64_t>(start[r0 + i], len), hi = std::min<uint64_t>(end[r0 + i], len);   // clipped to the sequence
                pos[i] = make_uint2(ix->anchor[sq] + (uint32_t)lo, ix->anchor[sq] + (uint32_t)hi);
            }
            BSX_CUDA_CHECK(cudaMemcpy(d_pos, pos.data(), (size_t)k * 8, cudaMemcpyHostToDevice));
            mhl_span_kernel<<<(k + 1 + 255) / 256, 256>>>(ix->d_refcat, m->d_cpg_rank, d_pos, k, d_span, d_chunks);
            BSX_CUDA_CHECK(cudaGetLastError());
            int rc = scan_exclusive(d_chunks, (uint64_t)k + 1); if (rc) return rc;
            uint32_t total = 0;
            BSX_CUDA_CHECK(cudaMemcpy(&total, d_chunks + k, 4, cudaMemcpyDeviceToHost));
            BSX_CUDA_CHECK(cudaMemset(d_out, 0, (size_t)k * 48 * 8));
            if (total) {
                const unsigned blocks = (unsigned)std::min<unsigned long long>((total + 7) / 8, (unsigned long long)std::max(per_sm, 1) * (unsigned)sms);
                meth_mhl_region_kernel<<<blocks, 256>>>(m->d_mhl, cuts ? d_cut : nullptr, d_chunks, d_span, k, d_out);
                BSX_CUDA_CHECK(cudaGetLastError());
            }
            BSX_CUDA_CHECK(cudaMemcpy(out + r0 * 48, d_out, (size_t)k * 48 * 8, cudaMemcpyDeviceToHost));
            BSX_CUDA_CHECK(cudaMemcpy(span.data(), d_span, (size_t)k * 8, cudaMemcpyDeviceToHost));
            for (uint32_t i = 0; i < k; i++) sites[r0 + i] = span[i].y - span[i].x;
        }
        return BSX_OK;
    };
    const int err = run();
    cudaFree(d_chunks); cudaFree(d_pos); cudaFree(d_span); cudaFree(d_out); cudaFree(d_cut);
    return err;
}

extern "C" size_t bsx_meth_write_mhl(bsx_meth *m, const bsx_meth_opts *o, uint64_t n, const uint32_t *seq, const uint64_t *start,
                                     const uint64_t *end, int fd) {
    if (!m || !o || (n && (!seq || !start || !end))) { bsx_set_error("bsx_meth_write_mhl: bad argument"); return 0; }
    if (!m->d_mhl) { bsx_set_error("bsx_meth_write_mhl: MHL was not enabled (bsx_meth_enable_mhl)"); return 0; }
    const bsx_index *ix = m->ix;
    const int threads = bsx_host_threads(0);
    size_t written = 0;
    auto put = [&](const std::string &s) {
        size_t off = 0;
        while (off < s.size()) { const ssize_t w = write(fd, s.data() + off, s.size() - off); if (w <= 0) return false; off += (size_t)w; written += (size_t)w; }
        return true;
    };
    if (!put("chr\tstart\tend\tsites\tcalls\tL\tMHL\tuMHL\thaplotypes\tmethylated\tunmethylated\n")) return 0;
    std::vector<uint64_t> sites, sums;
    for (uint64_t r0 = 0; r0 < n; r0 += MHL_SLICE) {
        const uint64_t k = std::min<uint64_t>(MHL_SLICE, n - r0);
        sites.resize(k); sums.resize(k * 48);
        if (bsx_meth_regions_mhl(m, o, k, seq + r0, start + r0, end + r0, sites.data(), sums.data()) != BSX_OK) return 0;
        std::vector<std::string> chunk((size_t)threads);
        bsx_parallel(threads, (size_t)k, [&](int t, size_t b, size_t e) {
            Sink s{&chunk[t]};
            for (size_t i = b; i < e; i++) {
                const uint64_t *T = &sums[i * 48], *M = T + BSX_MHL_MAX_LEN, *U = M + BSX_MHL_MAX_LEN;
                int L = 0;
                for (int l = 1; l <= BSX_MHL_MAX_LEN; l++) if (T[l - 1]) L = l;
                const std::string &name = ix->names[seq[r0 + i]];
                s.put(name.data(), name.size()); s.putc('\t'); s.putu(start[r0 + i]); s.putc('\t'); s.putu(end[r0 + i]); s.putc('\t');
                s.putu(sites[i]); s.putc('\t'); s.putu(T[0]); s.putc('\t'); s.putu((unsigned long long)L); s.putc('\t');
                if (!L) { s.put("NA\tNA\tNA\tNA\tNA\n", 15); continue; }
                // ascending l in double, as the oracle sums them
                double hm = 0.0, hu = 0.0;
                for (int l = 1; l <= L; l++) { hm += (double)((uint64_t)l * M[l - 1]) / (double)T[l - 1]; hu += (double)((uint64_t)l * U[l - 1]) / (double)T[l - 1]; }
                const double w = (double)(L * (L + 1) / 2);
                s.putf4(hm / w); s.putc('\t'); s.putf4(hu / w);
                for (const uint64_t *v : {T, M, U}) {
                    s.putc('\t');
                    for (int l = 1; l <= L; l++) { if (l > 1) s.putc(','); s.putu(v[l - 1]); }
                }
                s.putc('\n');
            }
        });
        for (const std::string &c : chunk) if (!put(c)) return 0;
    }
    return written;
}

int bsx_meth_write_mhl_file(bsx_meth *m, const bsx_meth_opts *o, const bsx_regions &rg, const char *path) {
    const int fd = open(path, O_WRONLY | O_CREAT | O_TRUNC, 0644);
    if (fd < 0) { fprintf(stderr, "failed to open MHL output file: %s\n", path); return BSX_ERR_IO; }
    const size_t w = bsx_meth_write_mhl(m, o, rg.seq.size(), rg.seq.data(), rg.start.data(), rg.end.data(), fd);
    close(fd);
    if (w == 0) { fprintf(stderr, "%s\n", bsx_last_error()); return BSX_ERR_IO; }
    uint64_t alignments = 0, calls = 0, valid = 0;
    if (bsx_meth_mhl(m, &alignments, &calls) != BSX_OK || bsx_meth_valid_count(m, &valid) != BSX_OK) { fprintf(stderr, "%s\n", bsx_last_error()); return BSX_ERR_CUDA; }
    fprintf(stderr, "MHL: %llu of %llu valid mappings carry a CpG call, %llu CpG calls in haplotypes\n", (unsigned long long)alignments,
            (unsigned long long)valid, (unsigned long long)calls);
    return BSX_OK;
}

// bsx_meth_regions, and with pdr != NULL bsx_meth_regions_pdr: one reduction fills both
static int meth_regions(bsx_meth *m, const bsx_meth_opts *o, uint64_t n, const uint32_t *seq, const uint64_t *start, const uint64_t *end,
                        uint64_t *out, uint64_t *pdr) {
    const bsx_index *ix = m->ix;
    for (uint64_t r = 0; r < n; r++) {
        if (seq[r] >= ix->n_seq) { bsx_set_error("bsx_meth_regions: region %llu: sequence %u of %u", (unsigned long long)r, seq[r], ix->n_seq); return BSX_ERR_ARG; }
        if (start[r] > end[r]) { bsx_set_error("bsx_meth_regions: region %llu: start %llu > end %llu", (unsigned long long)r, (unsigned long long)start[r],
                                               (unsigned long long)end[r]); return BSX_ERR_ARG; }
    }
    BSX_CUDA_CHECK(cudaSetDevice(ix->device));
    BSX_CUDA_CHECK(cudaDeviceSynchronize());           // in-process batches pile up on the mapper's streams
    int rc = combine_once(m, o); if (rc) return rc;
    if (n == 0) return BSX_OK;
    const uint64_t cap = std::min<uint64_t>(n, REGION_SLICE);
    unsigned long long *d_scan = nullptr, *d_out = nullptr, *d_pdr = nullptr; uint2 *d_span = nullptr;
    if (cudaMalloc(&d_scan, (cap + 1) * 8) != cudaSuccess || cudaMalloc(&d_span, cap * 8) != cudaSuccess || cudaMalloc(&d_out, cap * 12 * 8) != cudaSuccess ||
        (pdr && cudaMalloc(&d_pdr, cap * 2 * 8) != cudaSuccess)) {
        cudaGetLastError(); cudaFree(d_scan); cudaFree(d_span); cudaFree(d_out); bsx_set_error("bsx_meth_regions: out of device memory"); return BSX_ERR_CUDA; }
    int dev = 0, sms = 0, per_sm = 0;
    const int snp_mode = m->ct_snp == BSX_CT_SNP_SKIP || m->ct_snp == BSX_CT_SNP_CORRECT ? m->ct_snp : 0;
    const auto kern = region_kernel(o->combine_cpg != 0, snp_mode, pdr != nullptr);
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, 256, 0);
    const uint32_t min_depth = (uint32_t)std::max(o->min_depth, 1);
    std::vector<unsigned long long> scan;
    std::vector<uint2> span;
    int err = BSX_OK;
    for (uint64_t r0 = 0; r0 < n && err == BSX_OK; r0 += cap) {
        const uint32_t k = (uint32_t)std::min(cap, n - r0);
        scan.assign(k + 1, 0ull); span.resize(k);
        for (uint32_t i = 0; i < k; i++) {
            const uint32_t sq = seq[r0 + i], len = ix->size[sq];
            const uint64_t lo = std::min<uint64_t>(start[r0 + i], len), hi = std::min<uint64_t>(end[r0 + i], len);   // clipped to the sequence
            span[i] = make_uint2(ix->anchor[sq] + (uint32_t)lo, ix->anchor[sq] + (uint32_t)hi);
            scan[i + 1] = scan[i] + (hi - lo + REGION_CHUNK - 1) / REGION_CHUNK;
        }
        auto step = [&]() -> int {
            BSX_CUDA_CHECK(cudaMemcpy(d_scan, scan.data(), (k + 1) * 8, cudaMemcpyHostToDevice));
            BSX_CUDA_CHECK(cudaMemcpy(d_span, span.data(), (size_t)k * 8, cudaMemcpyHostToDevice));
            BSX_CUDA_CHECK(cudaMemset(d_out, 0, (size_t)k * 12 * 8));
            if (pdr) BSX_CUDA_CHECK(cudaMemset(d_pdr, 0, (size_t)k * 2 * 8));
            if (scan[k]) {
                const unsigned blocks = (unsigned)std::min<unsigned long long>((scan[k] + 7) / 8, (unsigned long long)std::max(per_sm, 1) * (unsigned)sms);
                kern<<<blocks, 256>>>(ix->d_refcat, m->d_meth, m->d_depth, m->d_confirm, m->d_snp, min_depth, d_scan, d_span, k, d_out, m->d_conc, m->d_disc, d_pdr);
                BSX_CUDA_CHECK(cudaGetLastError());
            }
            BSX_CUDA_CHECK(cudaMemcpy(out + r0 * 12, d_out, (size_t)k * 12 * 8, cudaMemcpyDeviceToHost));
            if (pdr) BSX_CUDA_CHECK(cudaMemcpy(pdr + r0 * 2, d_pdr, (size_t)k * 2 * 8, cudaMemcpyDeviceToHost));
            return BSX_OK;
        };
        err = step();
    }
    cudaFree(d_scan); cudaFree(d_span); cudaFree(d_out); cudaFree(d_pdr);
    return err;
}

extern "C" int bsx_meth_regions(bsx_meth *m, const bsx_meth_opts *o, uint64_t n, const uint32_t *seq, const uint64_t *start, const uint64_t *end,
                                uint64_t *out) {
    if (!m || !o || (n && (!seq || !start || !end || !out))) { bsx_set_error("bsx_meth_regions: bad argument"); return BSX_ERR_ARG; }
    return meth_regions(m, o, n, seq, start, end, out, nullptr);
}

extern "C" int bsx_meth_regions_pdr(bsx_meth *m, const bsx_meth_opts *o, uint64_t n, const uint32_t *seq, const uint64_t *start, const uint64_t *end,
                                    uint64_t *out, uint64_t *pdr) {
    if (!m || !o || (n && (!seq || !start || !end || !out || !pdr))) { bsx_set_error("bsx_meth_regions_pdr: bad argument"); return BSX_ERR_ARG; }
    if (!m->d_pdr) { bsx_set_error("bsx_meth_regions_pdr: PDR was not enabled (bsx_meth_enable_pdr)"); return BSX_ERR_ARG; }
    return meth_regions(m, o, n, seq, start, end, out, pdr);
}

extern "C" size_t bsx_meth_write_regions(bsx_meth *m, const bsx_meth_opts *o, uint64_t n, const uint32_t *seq, const uint64_t *start,
                                         const uint64_t *end, int fd) {
    if (!m || !o || (n && (!seq || !start || !end))) { bsx_set_error("bsx_meth_write_regions: bad argument"); return 0; }
    const bsx_index *ix = m->ix;
    static const char *const ctx[3] = {"CpG", "CHG", "CHH"};
    const int threads = bsx_host_threads(0);
    size_t written = 0;
    auto put = [&](const std::string &s) {
        size_t off = 0;
        while (off < s.size()) { const ssize_t w = write(fd, s.data() + off, s.size() - off); if (w <= 0) return false; off += (size_t)w; written += (size_t)w; }
        return true;
    };
    const bool pdr_on = m->d_pdr != nullptr;             // PDR: three more columns on every line
    if (!put(pdr_on ? "chr\tstart\tend\tcontext\tsites\tcovered\tC_count\tCT_count\tlevel\tconcordant\tdiscordant\tPDR\n"
                    : "chr\tstart\tend\tcontext\tsites\tcovered\tC_count\tCT_count\tlevel\n")) return 0;
    std::vector<uint64_t> sums, pdr;
    for (uint64_t r0 = 0; r0 < n; r0 += REGION_SLICE) {
        const uint64_t k = std::min<uint64_t>(REGION_SLICE, n - r0);
        sums.resize(k * 12); pdr.resize(k * 2);
        if (pdr_on ? bsx_meth_regions_pdr(m, o, k, seq + r0, start + r0, end + r0, sums.data(), pdr.data()) != BSX_OK
                   : bsx_meth_regions(m, o, k, seq + r0, start + r0, end + r0, sums.data()) != BSX_OK) return 0;
        std::vector<std::string> chunk((size_t)threads);
        bsx_parallel(threads, (size_t)k, [&](int t, size_t b, size_t e) {
            Sink s{&chunk[t]};
            for (size_t i = b; i < e; i++) {
                const std::string &name = ix->names[seq[r0 + i]];
                for (int c = 0; c < 3; c++) {
                    const uint64_t *v = &sums[(i * 3 + c) * 4];
                    s.put(name.data(), name.size()); s.putc('\t'); s.putu(start[r0 + i]); s.putc('\t'); s.putu(end[r0 + i]); s.putc('\t');
                    s.put(ctx[c], 3);
                    for (int f = 0; f < 4; f++) { s.putc('\t'); s.putu(v[f]); }
                    s.putc('\t');
                    if (v[3]) { char buf[48]; const int l = snprintf(buf, sizeof buf, "%.4f", (double)v[2] / (double)v[3]); s.put(buf, (size_t)l); }
                    else s.put("NA", 2);
                    if (pdr_on) {                                // the CpG line: the PDR file's lines in the region; CHG / CHH: none
                        const uint64_t pc = c == 0 ? pdr[i * 2] : 0, pd = c == 0 ? pdr[i * 2 + 1] : 0;
                        s.putc('\t'); s.putu(pc); s.putc('\t'); s.putu(pd); s.putc('\t');
                        if (pc + pd) { char buf[48]; const int l = snprintf(buf, sizeof buf, "%.4f", (double)pd / (double)(pc + pd)); s.put(buf, (size_t)l); }
                        else s.put("NA", 2);
                    }
                    s.putc('\n');
                }
            }
        });
        for (const std::string &c : chunk) if (!put(c)) return 0;
    }
    return written;
}

// name -> index of the selected sequences (a repeated name: the last record, as the command lines' own lookup)
static std::unordered_map<std::string, uint32_t> selected_names(const bsx_index *ix, const uint8_t *selected) {
    std::unordered_map<std::string, uint32_t> by;
    for (uint32_t k = 0; k < ix->n_seq; k++) if (!selected || selected[k]) by[ix->names[k]] = k;
    return by;
}

int bsx_regions_bed(const bsx_index *ix, const uint8_t *selected, const char *path, bsx_regions &rg) {
    rg = bsx_regions{};
    FILE *f = fopen(path, "rb");
    if (!f) { bsx_set_error("failed to open BED file: %s", path); return BSX_ERR_IO; }
    std::string text;
    char buf[1 << 16];
    for (size_t got; (got = fread(buf, 1, sizeof buf, f)) > 0;) text.append(buf, got);
    const bool io_err = ferror(f) != 0;
    fclose(f);
    if (io_err) { bsx_set_error("failed to read BED file: %s", path); return BSX_ERR_IO; }
    const auto by = selected_names(ix, selected);
    auto number = [](const char *p, const char *e, uint64_t &v) {
        if (p == e) return false;
        v = 0;
        for (; p < e; p++) {
            if (*p < '0' || *p > '9' || v > (UINT64_MAX - 9) / 10) return false;
            v = v * 10 + (uint64_t)(*p - '0');
        }
        return true;
    };
    uint64_t line = 0;
    for (size_t b = 0; b < text.size();) {
        size_t e = text.find('\n', b);
        if (e == std::string::npos) e = text.size();
        const size_t next = e + 1;
        line++;
        if (e > b && text[e - 1] == '\r') e--;
        const char *p = text.data() + b, *q = text.data() + e;
        b = next;
        if (std::all_of(p, q, [](char c) { return c == ' ' || c == '\t'; })) continue;
        auto starts = [&](const char *w) { const size_t l = strlen(w); return (size_t)(q - p) >= l && !memcmp(p, w, l) && ((size_t)(q - p) == l || p[l] == ' ' || p[l] == '\t'); };
        if (*p == '#' || starts("track") || starts("browser")) continue;
        const char *col[4] = {p, nullptr, nullptr, nullptr};
        int nc = 1;
        for (const char *x = p; x < q && nc < 4; x++) if (*x == '\t') col[nc++] = x + 1;
        if (nc < 3) { bsx_set_error("%s:%llu: fewer than 3 columns", path, (unsigned long long)line); return BSX_ERR_ARG; }
        const char *end3 = nc == 4 ? col[3] - 1 : q;
        uint64_t s = 0, t = 0;
        if (!number(col[1], col[2] - 1, s) || !number(col[2], end3, t)) {
            bsx_set_error("%s:%llu: start and end must be non-negative integers", path, (unsigned long long)line); return BSX_ERR_ARG; }
        if (s > t) { bsx_set_error("%s:%llu: start %llu > end %llu", path, (unsigned long long)line, (unsigned long long)s, (unsigned long long)t); return BSX_ERR_ARG; }
        const auto it = by.find(std::string(col[0], col[1] - 1));
        if (it == by.end()) { rg.skipped++; continue; }
        rg.seq.push_back(it->second); rg.start.push_back(s); rg.end.push_back(t);
    }
    return BSX_OK;
}

int bsx_regions_tiles(const bsx_index *ix, const uint8_t *selected, uint64_t width, bsx_regions &rg) {
    rg = bsx_regions{};
    if (width < 1) { bsx_set_error("tile width must be >= 1"); return BSX_ERR_ARG; }
    std::vector<uint32_t> order;
    for (uint32_t k = 0; k < ix->n_seq; k++) if (!selected || selected[k]) order.push_back(k);
    std::stable_sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return ix->names[a] < ix->names[b]; });   // the table's order
    for (uint32_t k : order)
        for (uint64_t s = 0; s < ix->size[k]; s += width) {
            rg.seq.push_back(k); rg.start.push_back(s); rg.end.push_back(std::min<uint64_t>(s + width, ix->size[k]));
        }
    return BSX_OK;
}

int bsx_meth_write_regions_file(bsx_meth *m, const bsx_meth_opts *o, const bsx_regions &rg, const char *path) {
    const int fd = open(path, O_WRONLY | O_CREAT | O_TRUNC, 0644);
    if (fd < 0) { fprintf(stderr, "failed to open region report file: %s\n", path); return BSX_ERR_IO; }
    const size_t w = bsx_meth_write_regions(m, o, rg.seq.size(), rg.seq.data(), rg.start.data(), rg.end.data(), fd);
    close(fd);
    if (w == 0) { fprintf(stderr, "%s\n", bsx_last_error()); return BSX_ERR_IO; }
    if (rg.skipped)
        fprintf(stderr, "regions: %llu of %llu skipped (sequence not in the reference or not selected)\n", (unsigned long long)rg.skipped,
                (unsigned long long)(rg.skipped + rg.seq.size()));
    return BSX_OK;
}
