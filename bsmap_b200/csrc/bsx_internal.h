// bsx_internal.h -- host-side structures behind the opaque C-ABI handles.
#pragma once
#include <cstdint>
#include <string>
#include <memory>
#include <vector>
#include <thread>
#include <cuda_runtime.h>
#include "../../include/bsmap_b200.h"

#define BSX_WIDE_CTX_V 8   // from this many allowed mismatches on, 32 context bases let too many candidates through (config 5)
struct bsx_block { uint32_t id, begin, end; };   // Block (dbseq.h:31-36)

// RefSeq (dbseq.h:59-114) as resident on one device
struct bsx_index {
    int device = -1;
    bsx_params par{};
    uint32_t n_seq = 0;
    std::vector<std::string> names;
    std::vector<uint32_t> size;        // title[2k].size
    std::vector<uint32_t> rc_offset;   // title[2k].rc_offset = 16 * nwords   (dbseq.cpp:225)
    std::vector<uint32_t> nwords;      // bfa[2k].n = ceil(len/16) + 2          (dbseq.cpp:60)
    std::vector<uint32_t> anchor;      // ref_anchor, n_seq + 1                  (dbseq.cpp:253-256)
    uint64_t n_words = 0, n_keys = 0, n_entries = 0;
    double build_seconds = 0;
    bool ref_only = false;             // packed strands only, no seed table (bsx_index_create_packed): cannot map
    // device arrays
    uint32_t *d_refcat = nullptr, *d_crefcat = nullptr;   // 2-bit packed strands, margins zeroed
    uint32_t *d_tab = nullptr;      // bsx_tab_len(): WGBS [2k] list start, [2k+1] start of rc part, [2k+2] end; RRBS CSR over (key, group)
    uint32_t *d_pos = nullptr;      // n_entries positions (ref_anchor + p), lists fwd-ascending then rc-ascending
    void *d_ctx = nullptr;          // inline context per entry: uint2 {the 16 reference bases before the seed, the 16 after it}, or,
                                    // when ctx_wide, uint4 {bases -32..-17, -16..-1, +s..+s+15, +s+16..+s+31}
    bool ctx_wide = false;          // WGBS index built with -v >= BSX_WIDE_CTX_V: 16-byte context entries
    uint32_t *d_tag = nullptr;      // RRBS: Hit.chr tag per entry
    uint32_t *d_seqinfo = nullptr;  // anchor[n_seq+1] | size[n_seq] | rc_offset[n_seq]
    uint32_t *d_sites = nullptr;    // RRBS: all digestion sites, concatenated
    uint32_t *d_site_off = nullptr; // RRBS: n_seq+1 offsets into d_sites
    // host copies used by the text formatter
    std::vector<uint32_t> h_refcat;                 // Watson strands (XR:Z / BSP refseq column)
    std::vector<std::vector<uint32_t>> sites;       // RRBS CCGG_sites (dbseq.cpp:158-163)
    std::vector<bsx_block> blocks;                  // WGBS: UnmaskRegion blocks, sorted (kept for bsx_index_save_packed)
};

// RRBS seed table: one CSR slot per (key, group), group = 2 * segment + mirrored (bsx_index.cu); dbseq.cpp:217 max_seedseg_num
static inline uint32_t bsx_rrbs_groups(int seed_size) { return 2u * (uint32_t)((10 - 1) * 16 / seed_size); }
// u32 entries of the table: WGBS [2k] list start, [2k+1] start of the rc half, [2k+2] end; RRBS [k * groups + g] group start
static inline uint64_t bsx_tab_len(const bsx_index *ix) {
    return ix->par.rrbs ? ix->n_keys * bsx_rrbs_groups(ix->par.seed_size) + 1 : 2 * ix->n_keys + 1;
}

static inline size_t bsx_ctx_entry_bytes(const bsx_index *ix) { return ix->ctx_wide ? 16 : 8; }

struct bsx_mapper;

// ---- host ingest / emit (bsx_reads.cpp, bsx_format.cpp) ----
struct bsx_view { const char *p; uint32_t n; };

// ReadClass (reads.h:26-48) over a memory-mapped FASTA / FASTQ file
struct bsx_reads {
    int fd = -1;
    const char *p = nullptr; size_t n = 0; bool mapped = false;
    // Streamed inputs (gzip'ed text, pipes): p / n / pos describe a WINDOW of the inflated stream, refilled as the
    // cutter advances (bsx_reads.cpp: stream_ensure); `keep` holds every window the current batch's views point into, so
    // a pipeline that moves the views on (bsx_cli.cpp: take_views) moves `keep` with them.  Memory stays bounded by the
    // batches in flight, whatever the size of the file.
    void *gz = nullptr;                    // gzFile; reads plain data transparently
    bool stream_eof = true;                // nothing left to inflate (always true for mapped files)
    bool io_error = false;                 // the stream ended in an error (corrupt or truncated gzip): what was read so far is served, the caller asks bsx_reads_failed
    bool win_starts_line = true;           // the window's first byte follows a line feed
    std::shared_ptr<std::vector<char>> win;
    std::vector<std::shared_ptr<std::vector<char>>> keep;
    size_t pos = 0;
    int kind = 0;                          // _file_format: 0 FASTQ, 1 FASTA, 3 BAM
    int readset = 0;                       // BAM: 0 single-end, 1 / 2 = file a / b of a pair (interleaved mates)
    int zero_qual = '!', max_readlen = BSX_MAX_READLEN;
    bool force_slow = false;
    std::vector<bsx_view> name, seq, qual; // the current batch
    std::vector<std::string> slow_store;   // backing store of records that took the token reader
    std::string qual_fill;                 // FASTA reads: zero_qual + default_qual (reads.cpp:108)
    std::vector<uint64_t> lines;
    std::vector<std::vector<uint64_t>> scan_parts;   // per-thread line starts of the current window (kept for their capacity)
    double rec_bytes = 0;                  // running bytes per record: sizes the next scan window
    uint64_t n_fast = 0, n_slow = 0;
};

// run f(tid, begin, end) over [0, n) on `threads` host threads (contiguous ranges)
template <class F> inline void bsx_parallel(int threads, size_t n, F f);

// formatter cores over (pointer, length) views; text is appended to one string per contiguous chunk
void bsx_format_se_chunks(const bsx_index *ix, const bsx_params *p, uint32_t n, const bsx_view *names, const bsx_view *seqs,
                          const bsx_view *quals, int readset, const bsx_rec *recs, const uint16_t *counts, int threads,
                          std::vector<std::string> &chunks, uint32_t *n_aligned);
void bsx_format_pe_chunks(const bsx_index *ix, const bsx_params *p, uint32_t n, const bsx_view *names_a, const bsx_view *seqs_a,
                          const bsx_view *quals_a, const bsx_view *names_b, const bsx_view *seqs_b, const bsx_view *quals_b,
                          const bsx_pair_rec *pr, const bsx_rec *ra, const bsx_rec *rb, const uint16_t *counts_a,
                          const uint16_t *counts_b, int threads, std::vector<std::string> &chunks,
                          std::vector<std::string> &chunks_unpair, uint32_t *n_stats);
int bsx_load_fasta(const char *path, std::vector<std::string> &names, std::vector<std::string> &seqs);   // bsx_reads.cpp
struct bsx_meth;
int bsx_meth_pile_mapped(bsx_meth *m, const bsx_meth_opts *o, int sam, int report_repeat_hits, uint32_t n, int mates, int readset, uint32_t stride,
                         const uint8_t *seq_a, const uint8_t *seq_b, const bsx_rec *out_a, const bsx_rec *out_b, const bsx_pair_rec *out_pair,
                         cudaStream_t st);   // bsx_meth.cu
// the command lines' M-bias output: bsx_meth_write_mbias to a new file at path, a warning on stderr for calls past
// BSX_MBIAS_CYCLES; errors are printed (bsx_meth.cu)
int bsx_meth_write_mbias_file(bsx_meth *m, const char *path);
// the command lines' conversion filter output: bsx_meth_write_conversion to a new file at path (NULL: no report), and
// on stderr "conversion filter: D of V valid mappings dropped (>= N methylated non-CpG calls)", or "(report only)" for
// N = 0; errors are printed (bsx_meth.cu)
int bsx_meth_write_conversion_file(bsx_meth *m, const char *path);
// the regions of the command lines' region report: (sequence, start, end) as given; `skipped` counts the BED regions on a
// sequence that is not in the reference or not selected (bsx_meth.cu)
struct bsx_regions { std::vector<uint32_t> seq; std::vector<uint64_t> start, end; uint64_t skipped = 0; };
// BED columns 1-3 against ix's names, the sequences with selected[k] != 0 (NULL = all); further columns, '#' / track /
// browser / blank lines are ignored, CRLF is accepted; fewer than 3 columns, a coordinate that is not a non-negative
// integer and start > end are errors naming the line (BSX_ERR_ARG; BSX_ERR_IO when the file cannot be read)
int bsx_regions_bed(const bsx_index *ix, const uint8_t *selected, const char *path, bsx_regions &rg);
// tiles [i*W, min((i+1)*W, len)) over every selected sequence, sequences sorted by name (the table's order)
int bsx_regions_tiles(const bsx_index *ix, const uint8_t *selected, uint64_t width, bsx_regions &rg);
// the region report (bsx_meth_write_regions) to a new file at path, and "regions: S of R skipped (...)" on stderr when
// the BED named sequences that are not there; errors are printed
int bsx_meth_write_regions_file(bsx_meth *m, const bsx_meth_opts *o, const bsx_regions &rg, const char *path);
// the command lines' PDR output: bsx_meth_write_pdr to a new file at path, and on stderr "PDR: I of V valid mappings
// informative (>= K CpG calls), D discordant"; errors are printed (bsx_meth.cu)
int bsx_meth_write_pdr_file(bsx_meth *m, const bsx_meth_opts *o, const char *const *seqs, const uint32_t *lens, const uint8_t *chroms, int threads,
                            const char *path);
// the command lines' epiallele output: bsx_meth_write_epialleles to a new file at path, and on stderr "epialleles: S of V
// valid mappings span a 4-CpG window, W window patterns counted"; errors are printed (bsx_meth.cu)
int bsx_meth_write_epialleles_file(bsx_meth *m, const bsx_meth_opts *o, const char *const *seqs, const uint32_t *lens, const uint8_t *chroms, int threads,
                                   const char *path);
// the command lines' MHL output: bsx_meth_write_mhl over the regions to a new file at path, and on stderr "MHL: A of V
// valid mappings carry a CpG call, C CpG calls in haplotypes"; errors are printed (bsx_meth.cu)
int bsx_meth_write_mhl_file(bsx_meth *m, const bsx_meth_opts *o, const bsx_regions &rg, const char *path);
// "no-action" / "correct" / "skip" -> BSX_CT_SNP_*, anything else 0 (bsx_meth.cu)
int bsx_ct_snp_mode(const char *name);
int bsx_inflate_file(const char *path, std::vector<char> &out);   // gzip / BGZF members -> bytes (bsx_reads.cpp)
int bsx_host_threads(int requested);   // 0 = BSX_THREADS env or hardware concurrency (capped at 32)

int bsx_index_build_device(bsx_index *ix, const char *const *seqs, const uint32_t *packed = nullptr);   // bsx_index.cu
int bsx_index_alloc_device(bsx_index *ix);                            // shell: allocate device arrays
void bsx_index_free_device(bsx_index *ix);
void bsx_set_error(const char *fmt, ...);

template <class F> inline void bsx_parallel(int threads, size_t n, F f) {
    if (threads < 1) threads = 1;
    if ((size_t)threads > n) threads = n ? (int)n : 1;
    if (threads == 1) { f(0, (size_t)0, n); return; }
    std::vector<std::thread> th;
    th.reserve(threads);
    for (int t = 0; t < threads; t++) {
        const size_t b = n * (size_t)t / threads, e = n * (size_t)(t + 1) / threads;
        th.emplace_back([=]() { f(t, b, e); });
    }
    for (auto &x : th) x.join();
}
