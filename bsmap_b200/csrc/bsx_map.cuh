// bsx_map.cuh -- kernel argument block and shared-memory layout of the mapping kernels.
#pragma once
#include "bsx_common.cuh"
#include "../../include/bsmap_b200.h"

#define BSX_MAX_KEYS 144          // seed_array[144] (align.h:84)
#define BSX_WARPS_PER_CTA 8       // warps of a mapping CTA; parameter sets whose per-warp shared memory is too large for eight run with 4, 2 or 1
#define BSX_MAX_CTA_SMEM (227u * 1024u)

struct MapArgs {
    // RefSeq
    const uint32_t *refcat, *crefcat, *tab, *pos, *tag, *seqinfo;
    const void *ctx;              // inline context per entry: uint2 {16 bases before, 16 after the seed}; wide indexes (-v >= BSX_WIDE_CTX_V):
                                  // uint4 {bases -32..-17, -16..-1, +s..+s+15, +s+16..+s+31}   // seqinfo: anchor[n+1] | size[n] | rc_offset[n]
    int ctx_wide;                 // 1: 16-byte context entries (the wide kernels)
    const uint32_t *sites, *site_off;
    uint32_t n_seq;
    // Param
    int s, I, v, W, r, min_insert, max_insert, chains, pairend, rrbs, randseed, max_ns, max_readlen;
    int n_adapter, site_len, digest_pos;
    uint32_t seed_bits;
    uint32_t rrbs_groups;         // RRBS: CSR slots per key of the seed table (bsx_rrbs_groups)
    int plan_cap;                 // plan entries per chain = max segments * I
    int nslot;                    // chains a read can use at once: 2 with -n 1, else 1 (plan storage per read)
    uint32_t read_smem, warp_smem_se, chain_stride, flank_off;   // derived from the two above on the host (bsx_map_args_derive)
    uint32_t img_slot, img_bytes; // prepared image in global scratch: ImgHdr + nslot x img_slot bytes
    int adapter_len[BSX_MAX_ADAPTERS];
    char adapter[BSX_MAX_ADAPTERS][64];
    char digest_site[32];
    // batch
    const uint8_t *seq_a, *seq_b;
    const uint16_t *len_a, *len_b;
    uint32_t stride, n, first_index;
    int readset;
    int packed;                   // 1: read slots hold 2-bit bases + valid mask (bsx_packed_stride), `stride` is the packed slot size
    uint32_t pk_mask_off, pk_maxlen;   // byte offset of the mask inside a packed slot; bases a slot can hold
    bsx_rec *out_a, *out_b;
    bsx_pair_rec *out_pair;
    uint16_t *cnt_a, *cnt_b;
    // scratch (global)
    uint32_t *work_counter;
    unsigned long long *stats;    // bsx_stats as 8 x u64
    uint2 *hit_scratch;           // per warp: reads_per_warp * hit_stride Hit{chr, loc}
    uint32_t *dd_scratch;         // per warp: reads_per_warp * dd_stride dedupe keys
    uint4 *pair_scratch;          // per warp: PE pair buckets
    uint32_t hit_stride, dd_stride, pair_stride;
    uint32_t *debug;              // optional: per read 40 u32 of seed-selection state (tests)
    uint8_t *prep;                // prepared-unit images: [warp][32] x img_bytes (bsx_prep.cuh)
    int mates;                    // units per read: 1 (SE) or 2 (PE)
    uint32_t block_units;         // units a warp prepares per work-counter atomic: 32, fewer for small batches (balance)
};

// One prepared read as the prepare phase (one THREAD per read: trim, filter, pack, choose seeds -- bsx_prep.cuh) leaves
// it in global scratch: this header, then per chain slot the packed read rw[10] | m5[10] and uint4 plan[plan_cap]:
// {list start, rc start, list end, read offset | segment << 16}.  480 bytes at config 2 (the first design wrote the
// whole ReadSm + plan + flanks: 1 056 bytes, all of which went to HBM and back).
struct ImgHdr {
    uint32_t index;                   // read index (myrand)
    uint32_t geom;                    // len | rmsn << 8 | seedseg << 16 | (filtered | fc << 1 | cc << 2) << 24
    uint32_t aux;                     // raw length | readset << 8
    uint32_t pad;
};
static_assert(sizeof(ImgHdr) == 16, "image header is one uint4");

// The read a warp is aligning, in shared memory: expanded from the image by load_image.  Followed by
// uint4 plan[nslot][plan_cap] and uint4 flank[nslot][plan_cap][FW]: read bases / mask facing the inline context before
// (x,y) and after (z,w) the seed of each plan entry (FW = 1; wide indexes FW = 2: the inner 16+16 bases, then the outer).
struct ReadSm {
    uint32_t rw[2][BSX_FIXWORDS];     // 2-bit read, chain 0 = as is, 1 = reverse complement (bseq/cbseq)
    uint32_t m5[2][BSX_FIXWORDS];     // 01 per ACGT base (reg/creg & 0x5555...)
    uint16_t nh[16], nc[16];          // _cur_n_hit / _cur_n_chit
    // per-read state (SingleAlign members), warp-uniform
    int raw, seedseg, readset, filtered;
    uint32_t index;
    int len, rmsn, nw;                // read length after trimming, read_max_snp_num, packed words
    uint32_t thres;                   // snp_thres
    int fc, cc;                       // flag_chain / cflag_chain
    uint32_t dn;                      // dedupe entries
    int best;                         // lowest mismatch level that holds a hit
    uint32_t pad_[3];
};
static_assert(sizeof(ReadSm) % 16 == 0, "images are copied as uint4");

// per-warp scratch of the prepare phase: the packed read of each lane's unit, lane-interleaved (no bank conflicts)
struct PrepCol {
    uint32_t rw[BSX_FIXWORDS][32], m5[BSX_FIXWORDS][32];
};

static_assert(sizeof(PrepCol) >= 4 * 32 * 16, "the align phase stages list heads (4 lists x 32 uint4) in the idle PrepCol");

// per-warp scratch of the align kernels
struct SelSm {
    uint16_t npairs[32];              // PE: _cur_n_hits[2*MAXSNPS+1]
    uint32_t ctr[8];                  // work counters of this warp (bsx_stats order), flushed to global rarely
};

// per-CTA constant tables (no integer division in the per-read code)
struct CtaSm {
    uint8_t profA[16 * 16];           // Param::InitMapping profile[n][i].a (param.cpp:85-93)
    uint8_t segof[160], remof[160];   // p / seed_size, p % seed_size
    uint16_t chr_lut[264];            // int2hit: sequence that holds position g << 24 of the concatenated reference (257 used)
};
static_assert(sizeof(CtaSm) % 16 == 0, "per-warp shared memory follows CtaSm and holds uint4");

// half-steps (32 list entries) per staging round: 2 KB of 8-byte entries at 8; wide indexes stage 16-byte entries.  Longer
// rounds spread the per-round work (schedule, staging issue, wait) over more entries but cost shared memory and leave
// more of a short mode's round empty: measured per kernel family (paired-end, config 3: 8 -> 81.3, 12 -> 84.2, 16 -> 80.3 M pairs/s;
// single-end WGBS, config 2: 8 -> 356.3, 12 -> 355.4 M reads/s; single-end RRBS, config 4: 12 and 16 gain 2 % resident and lose 4-7 %
// end to end in 1 M-read sub-batches).  The kernels (bsx_map_impl.cuh) and the host's shared-memory sizing both read it here.
constexpr __host__ __device__ int bsx_round_hs(int pe, int /*rrbs: 8 either way*/, int wide) { return (pe && !wide) ? 12 : 8; }
// bytes of the per-warp staging area beyond the PrepCol it aliases (slot[HS*32] entries + HS schedule entries of 32 / 48 bytes)
static inline __host__ __device__ size_t bsx_stage_extra_bytes(int wide, int pe, int rrbs) {
    const size_t need = (size_t)bsx_round_hs(pe, rrbs, wide) * (wide ? 32u * 16u + 48u : 32u * 8u + 32u);
    return need > sizeof(PrepCol) ? ((need - sizeof(PrepCol) + 15u) & ~(size_t)15u) : 0u;
}
static inline __host__ __device__ size_t bsx_read_smem_bytes(int plan_cap, int nslot, int wide) {
    return sizeof(ReadSm) + (size_t)nslot * (size_t)plan_cap * (wide ? 3u : 2u) * sizeof(uint4);
}
static inline size_t bsx_warp_smem_bytes(int reads_per_warp, int plan_cap, int nslot, int wide, int rrbs) {
    return (size_t)reads_per_warp * bsx_read_smem_bytes(plan_cap, nslot, wide) + sizeof(SelSm) + sizeof(PrepCol) + bsx_stage_extra_bytes(wide, reads_per_warp == 2, rrbs);
}
static inline size_t bsx_cta_smem_bytes(int reads_per_warp, int plan_cap, int nslot, int wide, int rrbs, int warps) {
    return sizeof(CtaSm) + bsx_warp_smem_bytes(reads_per_warp, plan_cap, nslot, wide, rrbs) * (size_t)warps;
}

static inline void bsx_map_args_derive(MapArgs &a) {
    a.read_smem = (uint32_t)bsx_read_smem_bytes(a.plan_cap, a.nslot, a.ctx_wide);
    a.warp_smem_se = (uint32_t)bsx_warp_smem_bytes(1, a.plan_cap, a.nslot, a.ctx_wide, a.rrbs);
    a.chain_stride = a.nslot == 2 ? (uint32_t)a.plan_cap : 0u;
    a.flank_off = (uint32_t)(a.nslot * a.plan_cap);
    a.img_slot = (uint32_t)(2 * BSX_FIXWORDS * 4 + a.plan_cap * sizeof(uint4));
    a.img_bytes = (uint32_t)(sizeof(ImgHdr) + a.nslot * a.img_slot);
}
static inline size_t bsx_image_bytes(int plan_cap, int nslot) {
    return sizeof(ImgHdr) + (size_t)nslot * (2 * BSX_FIXWORDS * 4 + (size_t)plan_cap * sizeof(uint4));
}

