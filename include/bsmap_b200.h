/* bsmap_b200.h -- C ABI of the B200-native BSMAP hot path (libbsmap_b200.so).
 *
 * The reference (BSMAP 2.6) has no plugin/FFI interface; the seam this ABI slots into is the three
 * calls a reference worker thread makes (main.cpp:49-114):
 *
 *     RefSeq::Run_ConvertBinseq + RefSeq::CreateIndex      (dbseq.cpp:215, 516)   -> bsx_index_create
 *     SingleAlign::ImportBatchReads + SingleAlign::Do_Batch (align.cpp:42, 591)   -> bsx_map_se (+ bsx_format_se)
 *     PairAlign::ImportBatchReads + PairAlign::Do_Batch     (pairs.cpp:27, 192)   -> bsx_map_pe (+ bsx_format_pe)
 *
 * Everything is `extern "C"`, plain pointers and sizes, opaque handles, int status codes
 * (0 = ok, non-zero = error; text via bsx_last_error()).  There is no CPU fallback: every compute
 * entry point fails with BSX_ERR_CUDA when no CUDA device is usable.
 *
 * Data layout
 *   reads   : ASCII, one read per `stride` bytes (stride % 8 == 0, stride >= 16 and >= longest read), plus
 *             uint16 lengths.  Reads longer than max_readlen are truncated (reads.cpp:115-117).
 *   records : fixed-size bsx_rec / bsx_pair_rec, the decision StringAlign / StringAlignPair makes
 *             before any text is produced; text formatting (s_OutHit & co) is host code in the same
 *             library (bsx_format_*), so names and qualities never travel to the device.
 */
#ifndef BSMAP_B200_H
#define BSMAP_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BSX_MAXSNPS 15        /* param.h:27  MAXSNPS              */
#define BSX_MAXHITS 1000      /* makefile:4  -DMAXHITS=1000       */
#define BSX_MAX_READLEN 144   /* param.h:23-25, param.cpp:80 (READ_144) */
#define BSX_MAX_ADAPTERS 10   /* param.h:99 */

enum { BSX_OK = 0, BSX_ERR_ARG = 1, BSX_ERR_CUDA = 2, BSX_ERR_NOMEM = 3, BSX_ERR_UNSUPPORTED = 4, BSX_ERR_IO = 5 };

/* Mirror of the option fields of class Param (param.h:54-121) that reach the hot path. */
typedef struct bsx_params {
    int32_t seed_size;          /* -s */
    int32_t index_interval;     /* -I */
    int32_t max_snp_num;        /* -v */
    int32_t max_num_hits;       /* -w */
    int32_t report_repeat_hits; /* -r */
    int32_t min_insert;         /* -m */
    int32_t max_insert;         /* -x */
    int32_t chains;             /* -n */
    int32_t pairend;            /* -b given */
    int32_t rrbs;               /* -D given */
    int32_t randseed;           /* -S */
    int32_t max_ns;             /* -f */
    int32_t max_readlen;        /* -L */
    int32_t out_sam;            /* -o *.sam */
    int32_t out_unmap;          /* -u */
    int32_t out_ref;            /* -R */
    int32_t digest_pos;         /* -D: index of '-' */
    int32_t n_adapter;          /* -A (repeatable) */
    char    digest_site[32];    /* -D with '-' removed */
    char    adapter[BSX_MAX_ADAPTERS][64];
} bsx_params;

/* Param::Param defaults (param.cpp:6-83) */
void bsx_params_default(bsx_params *p);

/* One record per read: what SingleAlign::StringAlign (align.cpp:610-627) decides. */
typedef struct bsx_rec {
    uint32_t loc;     /* Hit.loc, 0-based on the Watson strand            */
    uint32_t chr;     /* Hit.chr = 2*sequence + strand                     */
    uint32_t nhits;   /* hits in the lowest non-empty mismatch bucket      */
    uint8_t  nm;      /* that bucket's mismatch count                      */
    uint8_t  chain;   /* 0: read as is, 1: reverse-complemented read       */
    uint8_t  status;  /* 0: alignment attempted, 1: rejected by FilterReads */
    uint8_t  len;     /* read length after adapter trimming                */
} bsx_rec;

/* One record per pair: PairAlign::StringAlignPair (pairs.cpp:222-242). */
typedef struct bsx_pair_rec {
    uint32_t a_loc, a_chr, b_loc, b_chr;
    int32_t  insert;
    uint32_t npairs;
    uint8_t  na, nb, chain;
    uint8_t  paired;  /* 1: s_OutHitPair path; 0: the two bsx_rec of the mates apply (StringAlignUnpair) */
} bsx_pair_rec;

typedef struct bsx_index_info {
    uint64_t n_words;    /* u32 words per strand array incl. 2*400 margin words (dbseq.h:15) */
    uint64_t n_keys;     /* 3^seed_size (dbseq.cpp:314)                                      */
    uint64_t n_entries;  /* seed-table entries, both strands                                 */
    uint32_t n_seq;
    int32_t  device;
    double   build_seconds;   /* device time of pack + key + sort + table kernels */
    uint64_t n_tab;      /* u32 entries of the seed table: 2*n_keys+1 (WGBS), n_keys*groups+1 (RRBS, see below) */
    uint32_t ctx_words;  /* u32 per inline-context entry: 2, or 4 for a WGBS index built with -v >= 8             */
    uint32_t pad_;
} bsx_index_info;

/* work counters accumulated by the mapping kernels (SURVEY.md 8(d)) */
typedef struct bsx_stats {
    uint64_t candidates;      /* C: CountMismatch calls the reference semantics make      */
    uint64_t probes;          /* P: distinct seed-table headers read                      */
    uint64_t overfetch;       /* candidates evaluated speculatively past an exit point    */
    uint64_t full_extensions; /* candidates whose whole window was loaded (exact CountMismatch)  */
    uint64_t commits;         /* accepted hits                                            */
    uint64_t mapped;          /* reads / pairs with a reported location                   */
    uint64_t list_entries;    /* position-list entries loaded                             */
    uint64_t gathers;         /* candidates that survived the inline-context filter (one 16-byte HBM gather each) */
} bsx_stats;

typedef struct bsx_index bsx_index;     /* device-resident 2-bit reference + seed table (RefSeq) */
typedef struct bsx_mapper bsx_mapper;   /* per-device working set: batch buffers, scratch, streams */
typedef struct bsx_reads bsx_reads;     /* one FASTA / FASTQ read file (ReadClass, reads.h:26-48) */
typedef struct bsx_meth bsx_meth;       /* per-position methylation counters on one device (methratio.py:90-93) */

const char *bsx_last_error(void);
int bsx_device_count(void);

/* --- RefSeq::Run_ConvertBinseq + CreateIndex (dbseq.cpp:215-282, 516-523) ------------------- */
int bsx_index_create(const bsx_params *p, int n_seq, const char *const *names,
                     const char *const *seqs, const uint32_t *lens, int device, bsx_index **out);
int bsx_index_create_from_fasta(const bsx_params *p, const char *fasta_path, int device, bsx_index **out);
/* host-only index for the text layer (bsx_format_*): no device arrays, cannot map */
int bsx_index_create_text_only(const bsx_params *p, int n_seq, const char *const *names,
                               const char *const *seqs, const uint32_t *lens, bsx_index **out);
/* Packed reference cache (WGBS): the packed forward strand, UnmaskRegion blocks, names and sizes -- everything the
 * 0.4 s device rebuild of the seed table needs, without parsing the FASTA again.  Independent of -s / -I. */
int bsx_index_save_packed(const bsx_index *ix, const char *path);
int bsx_index_create_from_packed(const bsx_params *p, const char *path, int device, bsx_index **out);
/* packed reference only (no seed table): enough for bsx_meth, cannot map */
int bsx_index_create_packed(int n_seq, const char *const *names, const char *const *seqs, const uint32_t *lens,
                            int device, bsx_index **out);
int bsx_index_create_text_only_from_fasta(const bsx_params *p, const char *fasta_path, bsx_index **out);
int bsx_index_destroy(bsx_index *ix);
int bsx_index_get_info(const bsx_index *ix, bsx_index_info *info);
/* name/size of sequence k (RefTitle, dbseq.h:24-30) */
const char *bsx_index_seq_name(const bsx_index *ix, uint32_t k);
uint32_t bsx_index_seq_size(const bsx_index *ix, uint32_t k);
/* copy a device array to the host (parity tests): what = 0 refcat, 1 crefcat, 2 anchors (n_seq+1),
 * 3 tab (info.n_tab), 4 pos (n_entries), 5 RRBS tags (n_entries), 6 inline context (n_entries x info.ctx_words u32:
 * the 16 reference bases before and the 16 after each entry's seed; WGBS indexes built with -v >= 8 hold four words per
 * entry -- bases -32..-17, -16..-1 before the seed, +0..+15, +16..+31 after it).
 * RRBS (-D): the reference keeps one list per key and SnpAlign skips the entries whose (segment, mirrored) tag is not
 * the mode's (dbseq.cpp:418-438, align.cpp:187,229).  Here every list is stored partitioned by that tag -- group g =
 * 2*segment + mirrored, each group in the reference's order -- and tab is the CSR over (key, group):
 * tab[key*groups + g] .. tab[key*groups + g + 1], groups = 2 * (144 / seed_size). */
int bsx_index_download(const bsx_index *ix, int what, void *dst, size_t bytes);
/* device pointers + byte sizes of the arrays a replica needs (one-time NVLink broadcast):
 * order refcat, crefcat, tab, pos, tag, ctx, (unused: NULL/0).  Returns the count written (cap >= 7). */
int bsx_index_device_buffers(const bsx_index *ix, void **ptrs, size_t *bytes, int cap);
/* replica on another device: allocates there and copies over NVLink with cudaMemcpyPeer */
int bsx_index_replicate(const bsx_index *src, int device, bsx_index **out);
/* replica shell on `device` from the source's serialised metadata; the caller then fills the device
 * buffers (bsx_index_device_buffers) with its own broadcast (NCCL) */
size_t bsx_index_meta_size(const bsx_index *ix);
int bsx_index_meta_export(const bsx_index *ix, void *dst, size_t bytes);
int bsx_index_create_shell(const void *meta, size_t bytes, int device, bsx_index **out);

/* --- SingleAlign / PairAlign ----------------------------------------------------------------- */
int bsx_mapper_create(const bsx_index *ix, const bsx_params *p, uint32_t max_batch, uint32_t stride,
                      bsx_mapper **out);
int bsx_mapper_destroy(bsx_mapper *m);

/* Do_Batch with HOST buffers (end to end: H2D, kernels, D2H; returns when `out` is valid).
 * n may exceed max_batch: the call pipelines sub-batches over two streams.
 * counts: optional n*16 uint16 per-level hit counts (BSP output), may be NULL. */
int bsx_map_se(bsx_mapper *m, uint32_t n, const char *seqs, const uint16_t *lens,
               uint32_t first_index, int readset, bsx_rec *out, uint16_t *counts);
int bsx_map_pe(bsx_mapper *m, uint32_t n, const char *seqs_a, const uint16_t *lens_a,
               const char *seqs_b, const uint16_t *lens_b, uint32_t first_index,
               bsx_pair_rec *out, bsx_rec *out_a, bsx_rec *out_b, uint16_t *counts_a, uint16_t *counts_b);

/* Packed read input: the same calls with 2-bit bases + a 1-bit valid mask instead of ASCII -- 40 bytes per 100-nt read
 * slot instead of 104, for callers whose host->device link is the limit (eight GPUs fed from one host).  What the
 * reference's ConvertBinaySeq (align.cpp:90-162) derives from the text is derived here on the host, once.
 * Slot layout (bsx_packed_stride(stride) bytes, `stride` = the mapper's ASCII slot size): ceil(stride/4) bytes of bases,
 * four per byte, first base in bits 7:6, codes A0 C1 G2 T3, 0 for anything else; then ceil(stride/8) bytes of mask,
 * eight bases per byte, first base in bit 7, set for ACGT/acgt; zero padded to a multiple of 4.
 * Exactness: identical records to the ASCII entry points, except that letter case is lost -- with adapter trimming
 * (-A / -D), whose comparison is case sensitive in the reference (align.cpp:376), reads holding lower-case bases must
 * go through the ASCII call; bsx_pack_reads reports how many such bases it met.  Adapters and the digestion site
 * must be upper-case ACGT for the packed calls (BSX_ERR_UNSUPPORTED otherwise). */
size_t bsx_packed_stride(uint32_t stride);
int bsx_pack_reads(uint32_t n, const char *seqs, uint32_t stride, const uint16_t *lens, uint8_t *packed,
                   uint64_t *n_lowercase, int threads);
int bsx_map_se_packed(bsx_mapper *m, uint32_t n, const uint8_t *packed, const uint16_t *lens,
                      uint32_t first_index, int readset, bsx_rec *out, uint16_t *counts);
int bsx_map_pe_packed(bsx_mapper *m, uint32_t n, const uint8_t *packed_a, const uint16_t *lens_a,
                      const uint8_t *packed_b, const uint16_t *lens_b, uint32_t first_index,
                      bsx_pair_rec *out, bsx_rec *out_a, bsx_rec *out_b, uint16_t *counts_a, uint16_t *counts_b);

/* Staged form (inputs resident in HBM; used for kernel-only timing and by pipelined callers).
 * n <= max_batch.  `stream` is a cudaStream_t (NULL = the mapper's own stream). */
int bsx_batch_upload(bsx_mapper *m, uint32_t n, const char *seqs_a, const uint16_t *lens_a,
                     const char *seqs_b, const uint16_t *lens_b, void *stream);
int bsx_batch_upload_packed(bsx_mapper *m, uint32_t n, const uint8_t *packed_a, const uint16_t *lens_a,
                            const uint8_t *packed_b, const uint16_t *lens_b, void *stream);
int bsx_batch_run_se(bsx_mapper *m, uint32_t n, uint32_t first_index, int readset, void *stream);
int bsx_batch_run_pe(bsx_mapper *m, uint32_t n, uint32_t first_index, void *stream);
int bsx_batch_download_se(bsx_mapper *m, uint32_t n, bsx_rec *out, uint16_t *counts, void *stream);
int bsx_batch_download_pe(bsx_mapper *m, uint32_t n, bsx_pair_rec *out, bsx_rec *out_a, bsx_rec *out_b,
                          uint16_t *counts_a, uint16_t *counts_b, void *stream);
int bsx_mapper_sync(bsx_mapper *m);
/* counters since the last reset; number of kernel launches issued by this mapper */
int bsx_mapper_stats(bsx_mapper *m, bsx_stats *out, int reset);
uint64_t bsx_mapper_launches(const bsx_mapper *m);

/* --- text: s_OutHit / s_OutHitPair / s_OutHitUnpair (align.cpp:631-765, pairs.cpp:288-498) ---- */
/* return bytes needed (excluding NUL); if <= cap the text is in `out`. */
size_t bsx_format_header(const bsx_index *ix, char *out, size_t cap);            /* main.cpp:405-413 */
size_t bsx_format_se(const bsx_index *ix, const bsx_params *p, uint32_t n, const char *const *names,
                     const char *const *seqs, const char *const *quals, int readset,
                     const bsx_rec *recs, const uint16_t *counts, char *out, size_t cap, uint32_t *n_aligned);
size_t bsx_format_pe(const bsx_index *ix, const bsx_params *p, uint32_t n,
                     const char *const *names_a, const char *const *seqs_a, const char *const *quals_a,
                     const char *const *names_b, const char *const *seqs_b, const char *const *quals_b,
                     const bsx_pair_rec *pr, const bsx_rec *ra, const bsx_rec *rb,
                     const uint16_t *counts_a, const uint16_t *counts_b,
                     char *out, size_t cap, char *out_unpair, size_t cap_unpair, size_t *n_unpair,
                     uint32_t *n_stats /* pairs, single a, single b */);

/* --- read files: ReadClass::CheckFile / LoadBatchReads (reads.cpp:13-119), FASTA and FASTQ ---- */
/* The file is memory-mapped; regular 2- / 4-line records are cut on `threads` host threads, anything
 * irregular (blank lines, indented headers, trailing tokens) goes through a token reader with the
 * reference's ifstream `>>` / getline semantics, so both give what the reference would load.
 * Errors: BSX_ERR_IO when the file cannot be opened, BSX_ERR_ARG for an unrecognisable format. */
int bsx_reads_open(const char *path, int zero_qual, int max_readlen, bsx_reads **out);
void bsx_reads_close(bsx_reads *r);
int bsx_reads_kind(const bsx_reads *r);                       /* 0 FASTQ, 1 FASTA, 3 BAM (_file_format) */
int bsx_reads_failed(const bsx_reads *r);                     /* 1: a streamed input (gzip, pipe) ended in an error -- corrupt or truncated; the
                                                               * reads before it were served, bsx_last_error() has the text */
/* BAM input (reads.cpp:120-143): 0 single-end; 1 / 2 = this reader is file a / b of a pair whose mates are interleaved
 * in one BAM (a takes a record and skips the next, b skips one and takes the next) */
void bsx_reads_set_readset(bsx_reads *r, int readset);
void bsx_reads_skip(bsx_reads *r, uint64_t n_reads);          /* -B: 4 (fq) / 2 (fa) lines per read (reads.cpp:56-66) */
void bsx_reads_force_token_reader(bsx_reads *r, int on);      /* tests: disable the line cutter */
/* load up to `want` reads; bases go to seqs[i*stride ..] (zero padded) and lens[i]; returns the count.
 * Names / bases / qualities of the batch stay addressable through bsx_reads_get until the next call. */
uint32_t bsx_reads_next(bsx_reads *r, uint32_t want, uint32_t stride, char *seqs, uint16_t *lens, int threads);
int bsx_reads_get(const bsx_reads *r, uint32_t i, const char **name, uint32_t *name_len,
                  const char **seq, uint32_t *seq_len, const char **qual, uint32_t *qual_len);
/* format the current batch of `a` (and `b`) on `threads` host threads and write it, in input order,
 * to file descriptor fd (fd_unpair: the BSP -2 file, or -1).  Returns bytes written to fd. */
size_t bsx_emit_se(const bsx_index *ix, const bsx_params *p, const bsx_reads *a, uint32_t n, int readset,
                   const bsx_rec *recs, const uint16_t *counts, int threads, int fd, uint32_t *n_aligned);
size_t bsx_emit_pe(const bsx_index *ix, const bsx_params *p, const bsx_reads *a, const bsx_reads *b, uint32_t n,
                   const bsx_pair_rec *pr, const bsx_rec *ra, const bsx_rec *rb,
                   const uint16_t *counts_a, const uint16_t *counts_b, int threads, int fd, int fd_unpair,
                   uint32_t *n_stats /* pairs, single a, single b */);

/* --- `-o out.bam` (main.cpp:466-473: the reference shells out to sam2bam.sh = samtools view -bS | sort | index) ---- */
/* SAM text (BSMAP's own output) -> coordinate-sorted BAM at bam_path plus bam_path.bai, encoded, ordered, blocked and
 * indexed the way samtools 0.1.7 does it; the BGZF blocks are deflated on `threads` host threads. */
int bsx_sam_to_sorted_bam(const char *sam_path, const char *bam_path, int threads);

/* --- methratio.py (methylation ratios from the mappings) on the device -------------------------- */
typedef struct bsx_meth_opts {   /* methratio.py:5-16 */
    int32_t unique;        /* -u  process only unique mappings / pairs                         */
    int32_t pair;          /* -p  process only properly paired mappings                        */
    int32_t meth0;         /* -z  report loci with zero methylation ratios                     */
    int32_t trim_fillin;   /* -t  trim N end-repairing fill-in nucleotides (default 2)         */
    int32_t combine_cpg;   /* -g  combine CpG methylation ratios on both strands               */
    int32_t min_depth;     /* -m  report loci with sequencing depth >= FOLD (default 1)        */
    int32_t rm_dup;        /* -r  remove duplicated reads: the first alignment (in the order given) per
                            *     (sequence, fragment end, direction) counts; +8 bytes of HBM per position */
} bsx_meth_opts;
#define BSX_METH_SECONDARY 1u   /* alignment flag: not a unique mapping (SAM 's' / BSP flag != UM)      */
#define BSX_METH_PROPER    2u   /* alignment flag: properly paired       (SAM 'P' / BSP insert != 0)    */
#define BSX_METH_SAM       4u   /* alignment came from SAM: mate-overlap removal applies (methratio.py:64) */
void bsx_meth_opts_default(bsx_meth_opts *o);
/* zeroed meth / depth counters (u32) for every position of the index's Watson strand */
int bsx_meth_create(const bsx_index *ix, bsx_meth **out);
int bsx_meth_destroy(bsx_meth *m);
/* pile up n alignments (methratio.py:30-118).  seqs: SEQ as printed in the SAM / BSP file, `stride` bytes apart;
 * chr: 0-based index of the reference sequence; pos: 0-based leftmost position; strand: bit 0 = first ZS
 * character is '-', bit 1 = second is '-'; insert: TLEN (SAM) / insert size (BSP); mate_pos: PNEXT - 1;
 * flags: BSX_METH_*.  All host arrays.  *n_valid accumulates the "valid mappings" of the script's summary. */
int bsx_meth_add(bsx_meth *m, const bsx_meth_opts *o, uint32_t n, const char *seqs, uint32_t stride,
                 const uint16_t *lens, const uint32_t *chr, const uint32_t *pos, const uint8_t *strand,
                 const int32_t *insert, const int32_t *mate_pos, const uint8_t *flags, uint64_t *n_valid);
/* In-process form: every batch `mp` maps from now on is piled up on the device right after the align kernel, from
 * the device-resident reads and records -- no SAM text in between.  Which reads count, with which SEQ orientation,
 * POS, TLEN and PNEXT, follows s_OutHit / s_OutHitPair / s_OutHitUnpair; sam_rules = 1 applies the script's SAM
 * branch (mate-overlap removal), 0 its BSP branch.  meth = NULL detaches.  The counters must live on mp's device. */
int bsx_mapper_attach_meth(bsx_mapper *mp, bsx_meth *meth, const bsx_meth_opts *o, int sam_rules);
int bsx_meth_valid_count(bsx_meth *m, uint64_t *n_valid);   /* "valid mappings" so far (synchronises the device) */
/* copy the counters of sequence k to the host (after -g combining when o->combine_cpg; idempotent) */
int bsx_meth_download(bsx_meth *m, const bsx_meth_opts *o, uint32_t k, uint32_t *meth, uint32_t *depth);
/* write the table of methratio.py:133-152 for the sequences selected by `chroms` (NULL = all), sorted by
 * name, to fd.  seqs / lens: the reference records as in bsx_index_create (needed for the context column).
 * stats: covered cytosines, their summed depth.  Returns bytes written. */
size_t bsx_meth_write(bsx_meth *m, const bsx_meth_opts *o, const char *const *seqs, const uint32_t *lens,
                      const uint8_t *chroms /* n_seq flags or NULL */, int threads, int fd, uint64_t *stats);
/* --- M-bias: methylation level by position in the read, and per-cycle exclusion of calls ----------
 * A call is one increment of the counters above (after -u / -p, -r, -t, mate-overlap removal and the bounds test).
 * Its cycle is its 0-based offset j in SEQ as printed, or L-1-j when SEQ is printed reversed (the two ZS characters
 * differ), L being the printed length; its read is 2 when the printed FLAG has 0x80 (bsx_meth_add: BSX_METH_READ2;
 * in process: mate b of bsx_map_pe, or readset 2 of bsx_map_se), else 1; its context is CpG / CHG / CHH from the
 * reference on the call's strand (non-ACGT and positions off the sequence count as H). */
#define BSX_METH_READ2     8u   /* alignment flag: read 2 (FLAG 0x80) -- M-bias and exclusion only       */
#define BSX_MBIAS_CYCLES   512  /* cycles tracked; calls at later cycles count in the table and in *overflow */
/* track M-bias from now on.  Must precede the first alignment piled up (BSX_ERR_ARG otherwise). */
int bsx_meth_enable_mbias(bsx_meth *m);
/* drop every call of read 1 with cycle < ignore[0] or cycle >= L - ignore[1], and of read 2 with cycle < ignore[2]
 * or cycle >= L - ignore[3], from the counters and from the M-bias ("valid mappings" and -r are unaffected).  All
 * zero (the default) drops nothing.  Must precede the first alignment piled up; negative values: BSX_ERR_ARG. */
int bsx_meth_set_ignore(bsx_meth *m, const int32_t ignore[4] /* r1_5p, r1_3p, r2_5p, r2_3p */);
/* the M-bias so far (synchronises the device): out has 2 x 3 x BSX_MBIAS_CYCLES x 2 counters, index
 * ((read * 3 + ctx) * BSX_MBIAS_CYCLES + cycle) * 2 + {0 methylated, 1 unmethylated} with read 0 / 1 = read 1 / 2 and
 * ctx 0 / 1 / 2 = CpG / CHG / CHH; *overflow (may be NULL): calls at cycle >= BSX_MBIAS_CYCLES.  BSX_ERR_ARG when
 * M-bias was not enabled. */
int bsx_meth_mbias(bsx_meth *m, uint64_t *out, uint64_t *overflow);
/* write the M-bias report to fd: a header line "context read cycle methylated unmethylated ratio" (tab-separated),
 * then per context CpG, CHG, CHH, per read 1, 2, per 1-based cycle ascending, a row when methylated + unmethylated
 * > 0, ratio = %.3f of methylated / (methylated + unmethylated).  Returns bytes written (0 on error). */
size_t bsx_meth_write_mbias(bsx_meth *m, int fd);
/* --- C/T SNP evidence from the opposite strand, and SNP-corrected ratios ---------------------------------------------
 * Bisulfite leaves the opposite strand's base untouched, so it tells a genomic T at a reference C (which reads like an
 * unmethylated C) from a real C.  Evidence bases are those of an alignment that survive every step a call survives
 * (-u / -p, -r, -t, mate-overlap removal, the bounds test, and bsx_meth_set_ignore's cycle rule); q = reference position.
 *   '+' alignment (first ZS character '+'), reference G at q: read G -> confirm[q] += 1, read A -> snp[q] += 1
 *   '-' alignment, reference C at q:                          read C -> confirm[q] += 1, read T -> snp[q] += 1
 * Other read characters count nothing (compared in upper case, as the calls are); non-ACGT reference bases count nothing.
 * Calls, the M-bias and "valid mappings" are unchanged.  -g adds a CpG's G evidence to its C and zeroes the G.
 * With the option set, bsx_meth_write writes 12 columns:
 *   chr pos strand context ratio eff_CT_count C_count CT_count rev_G_count rev_GA_count CI_lower CI_upper
 * with C_count = meth, CT_count = depth, rev_G_count = confirm, rev_GA_count = confirm + snp, over the lines the plain
 * table prints (depth >= min_depth, depth > 0, meth > 0 unless -z); the mode then sets eff or drops the line:
 *   BSX_CT_SNP_NO_ACTION  eff = CT
 *   BSX_CT_SNP_CORRECT    eff = CT when rev_GA == 0, else (double)CT * rev_G / rev_GA; the line is dropped when eff == 0
 *   BSX_CT_SNP_SKIP       the line is dropped when rev_G < rev_GA, else eff = CT
 * ratio = min(C, eff) / eff and the Wilson interval with eff for the depth; eff prints as %.2f.  The summary (covered
 * cytosines, their summed depth) is the plain table's in every mode.  8 more bytes of HBM per position. */
#define BSX_CT_SNP_NO_ACTION 1
#define BSX_CT_SNP_CORRECT   2
#define BSX_CT_SNP_SKIP      3
/* count the evidence from now on and write the 12-column table in `mode`.  Must precede the first alignment piled up;
 * a bad mode or a late call: BSX_ERR_ARG; no device memory for the two arrays: BSX_ERR_CUDA. */
int bsx_meth_enable_ct_snp(bsx_meth *m, int mode);
/* copy the evidence of sequence k to the host (after -g combining when o->combine_cpg, like bsx_meth_download);
 * BSX_ERR_ARG when the evidence was not enabled */
int bsx_meth_download_ct_snp(bsx_meth *m, const bsx_meth_opts *o, uint32_t k, uint32_t *confirm, uint32_t *snp);
/* --- conversion filter: drop incompletely bisulfite-converted alignments ---------------------------------------------
 * A fragment that bisulfite did not convert reads C at every C it covers, so its non-CpG Cs, almost never methylated
 * in mammals, look methylated.  The filter scores each alignment and drops those that look unconverted.
 *   call     one increment of the counters, after every other rule: -u / -p, -r, -t, mate-overlap removal, the bounds
 *            test and bsx_meth_set_ignore's cycle rule (excluded cycles, trimmed bases and the mate overlap hold none)
 *   context  the M-bias rule: a '+' C at q is CpG if q+1 is G, else CHG if q+2 is G, else CHH; a '-' G at q the same
 *            with q-1, q-2 and C; non-ACGT bases and positions off the sequence count as H
 *   score    the alignment's calls that are methylated (read C on '+', read G on '-') in CHG or CHH context
 *   filter   threshold N, 1 <= N <= 255: an alignment with score >= N adds nothing to meth / depth, the M-bias or the
 *            C/T SNP evidence; it is still a valid mapping (bsx_meth_valid_count and the summary line are unchanged).
 *            N = 0 drops nothing: the scores are only counted.  The filter is per alignment: each mate on its own calls.
 *   -r       the claim is decided before the filter: a dropped alignment still holds its (position, direction), so its
 *            later duplicates still lose (the outcome does not depend on how the alignments are cut into batches)
 *   report   a histogram of the valid mappings by score, BSX_CONV_BINS bins, bin b = score b, the last 255 or more; the
 *            bins sum to the valid mappings, and the dropped alignments are the bins >= N. */
#define BSX_CONV_BINS 256
/* score every alignment from now on and drop those scoring threshold or more (0..255; 0 = report only).  Must precede
 * the first alignment piled up; a bad threshold or a late call: BSX_ERR_ARG.  2 KB of device memory. */
int bsx_meth_enable_conversion_filter(bsx_meth *m, int32_t threshold);
/* the score histogram so far (synchronises the device): out has BSX_CONV_BINS counters; *dropped (may be NULL): the
 * alignments dropped.  BSX_ERR_ARG when the filter was not enabled. */
int bsx_meth_conversion(bsx_meth *m, uint64_t *out /* BSX_CONV_BINS */, uint64_t *dropped);
/* write the report to fd: a header line "methylated_nonCpG_calls alignments dropped" (tab-separated), then one row per
 * non-empty bin, ascending, the last labelled "255+"; dropped is 1 when the bin's alignments were dropped, else 0.
 * Returns bytes written (0 on error). */
size_t bsx_meth_write_conversion(bsx_meth *m, int fd);
/* --- read-level CpG concordance: the proportion of discordant reads (PDR) --------------------------------------------
 * A level of 0.5 at a CpG may come from half the molecules fully methylated and half unmethylated, or from every molecule
 * methylated at random.  PDR tells these apart by the CpG calls each read carries.
 *   call         one increment of the counters, after every other rule (as for the conversion filter): -u / -p, -r, -t,
 *                mate-overlap removal, the bounds test and bsx_meth_set_ignore's cycle rule
 *   context      the M-bias rule: a '+' C at q is CpG if q+1 is G; a '-' G at q is CpG if q-1 is C
 *   pattern      m = the alignment's methylated CpG calls, u = its unmethylated ones; a read character that is neither
 *                the methylated nor the converted letter (N, lower case) is no call.  Each mate on its own calls.
 *   informative  m + u >= K, 1 <= K <= 255 (default 4); an informative alignment is concordant when m == 0 or u == 0,
 *                else discordant
 *   counters     every CpG call of an informative alignment adds 1 to concordant[q] or discordant[q], by the alignment's
 *                class; other alignments add nothing.  -g adds a CpG's G counts to its C and zeroes the G.
 *   other rules  an alignment dropped by the conversion filter and a -r loser are not scored; calls, the M-bias, the C/T
 *                SNP evidence, the conversion histogram and "valid mappings" do not change
 *   summary      the informative alignments and the discordant ones
 *   file         header "chr pos strand concordant discordant PDR" (tab-separated), one line per position with
 *                concordant + discordant >= max(-m, 1) that the C/T SNP mode would not drop (BSX_CT_SNP_SKIP: any SNP
 *                evidence; BSX_CT_SNP_CORRECT: eff == 0), sequences selected and sorted by name, positions ascending;
 *                strand from the reference base as in the table; PDR = discordant / (concordant + discordant) as %.3f;
 *                -z is ignored
 *   regions      bsx_meth_write_regions adds the columns "concordant discordant PDR" to every line: on the CpG line the
 *                sums over the PDR file's lines in the region and PDR = %.4f (NA at 0), on the CHG and CHH lines 0 0 NA
 * 8 more bytes of HBM per position. */
/* score every alignment from now on; min_cpg = K.  Must precede the first alignment piled up; K outside 1..255 or a late
 * call: BSX_ERR_ARG; no device memory for the two arrays: BSX_ERR_CUDA. */
int bsx_meth_enable_pdr(bsx_meth *m, int32_t min_cpg);
/* copy the concordance counters of sequence k to the host (after -g combining when o->combine_cpg, like
 * bsx_meth_download); BSX_ERR_ARG when PDR was not enabled */
int bsx_meth_download_pdr(bsx_meth *m, const bsx_meth_opts *o, uint32_t k, uint32_t *concordant, uint32_t *discordant);
/* the informative and discordant alignments so far (synchronises the device; either may be NULL); BSX_ERR_ARG when PDR
 * was not enabled */
int bsx_meth_pdr(bsx_meth *m, uint64_t *informative, uint64_t *discordant);
/* write the PDR file to fd for the sequences selected by `chroms` (NULL = all); seqs / lens as in bsx_meth_write.
 * Returns bytes written (0 on error). */
size_t bsx_meth_write_pdr(bsx_meth *m, const bsx_meth_opts *o, const char *const *seqs, const uint32_t *lens,
                          const uint8_t *chroms /* n_seq flags or NULL */, int threads, int fd);
/* --- methylation levels over regions, reduced on the device from the counters ----------------------------------------
 *   region   (sequence, start, end), 0-based and half-open as in BED; start == end is empty; an end past the sequence end
 *            is clipped when counting.  Each region is reported for the contexts CpG, CHG, CHH (ctx 0, 1, 2).
 *   site     a reference C (strand '+') or G (strand '-') at a position q with start <= q < end.  Its context is the
 *            M-bias rule on its strand: '+' CpG if q+1 is G, else CHG if q+2 is G, else CHH; '-' the same with q-1, q-2
 *            and C; non-ACGT bases and positions off the sequence count as H.  With -g a G that follows a C is not a
 *            site: its counts sit on the C, and the CpG is one site.
 *   sites    the number of sites
 *   covered  the sites whose line the table would print with -z: depth >= max(-m, 1), and, with C/T SNP evidence, not
 *            dropped by the mode (BSX_CT_SNP_SKIP: any SNP evidence; BSX_CT_SNP_CORRECT: eff == 0)
 *   C, CT    over the covered sites, the sums of the table's methylated count (methy_C / C_count) and of its depth
 *            (total_C / the raw CT_count)
 * So covered, C and CT are the count and the sums of the -z table's lines in the region, by context.  -z itself is
 * ignored (leaving out unmethylated sites would bias the levels up), and `correct`'s scaled eff_CT_count is not summed:
 * the sums stay exact integers. */
/* out[(r * 3 + ctx) * 4 + {0 sites, 1 covered, 2 C, 3 CT}] for the n regions (seq: sequence index; a bad index or
 * start > end: BSX_ERR_ARG).  Synchronises the device.  -g combines the counters first, like bsx_meth_download; without
 * -g the counters are not changed, so more alignments may be added afterwards. */
int bsx_meth_regions(bsx_meth *m, const bsx_meth_opts *o, uint64_t n, const uint32_t *seq, const uint64_t *start, const uint64_t *end,
                     uint64_t *out);
/* write the region report to fd: a header line "chr start end context sites covered C_count CT_count level"
 * (tab-separated), then three lines per region, CpG, CHG, CHH, in region order, start and end as given; level = %.4f
 * of C / CT, or NA when CT == 0.  With PDR enabled, "concordant discordant PDR" follow on every line (see above).
 * Returns bytes written (0 on error). */
size_t bsx_meth_write_regions(bsx_meth *m, const bsx_meth_opts *o, uint64_t n, const uint32_t *seq, const uint64_t *start, const uint64_t *end,
                              int fd);
/* bsx_meth_regions, and pdr[r * 2 + {0 concordant, 1 discordant}]: the sums over the PDR file's lines in region r (with
 * PDR on, bsx_meth_write_regions adds them and their PDR to the report).  BSX_ERR_ARG when PDR was not enabled. */
int bsx_meth_regions_pdr(bsx_meth *m, const bsx_meth_opts *o, uint64_t n, const uint32_t *seq, const uint64_t *start, const uint64_t *end,
                         uint64_t *out, uint64_t *pdr);
/* the methratio.py command line: -o -d [-c -u -p -z -q -r -t -g -m -s] files... (SAM, BAM and BSP; -s is ignored);
 * extensions: --mbias FILE (the M-bias report) and --mbias-ignore A,B,C,D (bsx_meth_set_ignore), SAM and BAM only;
 * --ct-snp no-action|correct|skip (bsx_meth_enable_ct_snp); --conversion-filter N and --conversion-report FILE
 * (bsx_meth_enable_conversion_filter, bsx_meth_write_conversion); --region-report FILE with --regions BED or --tiles W
 * (bsx_meth_write_regions); --pdr FILE [--pdr-min-cpg K] (bsx_meth_enable_pdr, bsx_meth_write_pdr) */
int bsx_methratio_main(int argc, char **argv);

/* --- the bsmap command line (main.cpp:441-476): same options, same output files -------------- */
int bsx_cli_main(int argc, char **argv);
/* a stand-alone executable that will _exit() right after bsx_cli_main may skip the device teardown (1.8 s at 3.1 Gb) */
void bsx_cli_exit_after_main(int on);

#ifdef __cplusplus
}
#endif
#endif
