// bsx_map_impl.cuh -- SingleAlign / PairAlign on the device (align.cpp, align.h, pairs.cpp): the body of the six mapping
// kernels.  Each translation unit bsx_map_{se,pe}{,_rrbs,_wide}.cu describes its kernel in `struct MapKernel` (paired-end,
// RRBS, wide context, and the two schedule choices of the list walk) before it includes this file, then defines its
// __global__ with its own __launch_bounds__ around map_se() or map_pe().  The mode is a compile-time constant, so dead code
// leaves each binary, and everything is inlined with one call site per device function: the kernels are instruction-cache
// sensitive (paired-end: 117 -> 93 KB of SASS, no call spills).
//
// Warps are persistent and fetch work with an atomic counter.  A warp takes up to 32 units (reads, or mates of 16
// pairs) at a time:
//
//   phase A  prepare, one THREAD per unit (bsx_prep.cuh)
//     K2  trim / filter / pack   TrimAdapter, FilterReads, ConvertBinaySeq (align.cpp:371-425, 579-589, 90-162)
//     K3  seed selection         ReorderSeed / AdjustSeedStartArray / CountSeeds (align.cpp:454-577): every distinct
//                                read offset that can carry a seed is probed once; the plan of (mode, sub-seed) ->
//                                list bounds + the read words facing the inline context goes into the unit's image
//   phase B  align, one WARP per unit (this file): the image is copied into shared memory, then
//     K4  probe + extend + commit  SnpAlign + CountMismatch (align.cpp:253-346, align.h:167-200): 64 list entries
//                                per step, two per lane.  Phase 0 rejects a candidate from the 8 bytes of reference
//                                context stored next to its table entry (no random access); survivors get one aligned
//                                16-byte gather when a step has many of them, then the exact window count (few
//                                survivors: cooperatively, two per memory round trip).  Every phase is a lower bound
//                                of CountMismatch, so accept / reject decisions are the reference's.  Survivors are
//                                committed in list order (ballot + serial loop) so dedupe, bucket counts, -w threshold
//                                lowering and the -r 0 exits fire at exactly the candidate the sequential reference
//                                would stop at.
//     K5  selection              StringAlign (align.cpp:610-627) + myrand.
//     K6  pairing                PairAlign::RunAlign / GetPairs (pairs.cpp:34-190).
//
// Integer work bound by memory latency and issue slots: no tensor cores.
#include <type_traits>
#include "bsx_map.cuh"

#include "bsx_prep.cuh"

namespace {

constexpr int ROUND_HS = bsx_round_hs(MapKernel::pe, MapKernel::rrbs, MapKernel::wide);   // half-steps per staging round
constexpr int FW = MapKernel::wide ? 2 : 1;   // uint4 per plan entry in the flank array: wide indexes hold 32 + 32 context bases

// work counters live in shared memory (SelSm::ctr, bsx_stats order); lane 0 updates them
enum { CT_CAND = 0, CT_PROBE, CT_OVER, CT_FULL, CT_COMMIT, CT_MAPPED, CT_LIST, CT_GATHER };
typedef uint32_t Ctr;
// warp-uniform state in shared memory is written by lane 0 only, fenced on both sides
#define WSET(lhs, rhs) do { const auto v_ = (rhs); __syncwarp(); if (lane == 0) (lhs) = v_; __syncwarp(); } while (0)
#define CTR_ADD(C, k, v) do { const uint32_t v_ = (uint32_t)(v); if (lane == 0) (C)[k] += v_; } while (0)   // v may hold warp collectives

__device__ __forceinline__ uint4 *plan_of(ReadSm *R, int chain, const MapArgs &A) {
    return reinterpret_cast<uint4 *>(reinterpret_cast<uint8_t *>(R) + sizeof(ReadSm)) + chain * A.chain_stride;
}
__device__ __forceinline__ uint4 *flank_of(ReadSm *R, int chain, const MapArgs &A) {
    return reinterpret_cast<uint4 *>(reinterpret_cast<uint8_t *>(R) + sizeof(ReadSm)) + A.flank_off + chain * A.chain_stride * FW;
}

// 16 bases of the read from offset `off` (may start before the read or run past it): (bases, valid mask)
__device__ __forceinline__ uint2 read_window(const ReadSm *R, int chain, int off) {
    if (off <= -16 || off >= 16 * BSX_FIXWORDS) return make_uint2(0u, 0u);
    if (off < 0) return make_uint2(R->rw[chain][0] >> (2 * -off), R->m5[chain][0] >> (2 * -off));
    const int j = off >> 4, sh = (off & 15) * 2;
    const uint32_t r1 = (j + 1 < BSX_FIXWORDS) ? R->rw[chain][j + 1] : 0u, m1 = (j + 1 < BSX_FIXWORDS) ? R->m5[chain][j + 1] : 0u;
    return make_uint2(__funnelshift_l(r1, R->rw[chain][j], sh), __funnelshift_l(m1, R->m5[chain][j], sh));
}

// The read bases that face an entry's inline context are fixed per list, the context word varies per candidate.  With
// M = one bit per valid base (low) plus the high bit of every valid base that is not T, a base mismatches iff
// ((q ^ s) & M) has a bit in its field: read T (11) matches reference T and C (low bit equal), everything else must be
// equal -- the same decision as XM((q & XC(s)) ^ s) & r (param.h:126,139-147, bsx_mm_word_bits) in four instead of six
// operations per word, and the two words of a candidate share one popcount.
__device__ __forceinline__ uint32_t flank_mask(uint32_t q, uint32_t m5) { return m5 | ((m5 & ~(q & (q >> 1))) << 1); }
// f = {q before, M before, q after, M after}, c = {16 bases before the seed, 16 after}
__device__ __forceinline__ uint32_t ctx_mm2(const uint4 f, const uint2 c) {
    const uint32_t ub = (f.x ^ c.x) & f.y, ua = (f.z ^ c.y) & f.w;
    return (uint32_t)__popc(((ub | (ub >> 1)) & 0x55555555u) | ((ua | (ua << 1)) & 0xAAAAAAAAu));
}

// Asynchronous 16-byte copy global -> shared (LDGSTS, bypasses L1 and the register file): the warp requests the heads
// of all lists of a group back to back and waits once, instead of one DRAM round trip per list.  List heads and tails
// fetch 64-byte granules from HBM, not 128-byte lines.
__device__ __forceinline__ void cp_async16s(uint32_t smem_addr, const void *gsrc) {   // destination as a shared-window address
    asm volatile("cp.async.cg.shared.global.L2::64B [%0], [%1], 16;" :: "r"(smem_addr), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" :: "n"(N) : "memory"); }

__device__ __forceinline__ const CtaSm *cta_tables() {   // the CTA's tables sit at the start of dynamic shared memory
    extern __shared__ __align__(16) uint8_t bsx_dyn_smem_[];
    return reinterpret_cast<const CtaSm *>(bsx_dyn_smem_);
}

// per-CTA tables: seed profile and p -> (segment, remainder) for the prepare phase, the granule table for int2hit
__device__ __forceinline__ void init_cta_tables(const MapArgs &A, CtaSm *K) {
    #pragma unroll 1
    for (int t = threadIdx.x; t < 256; t += blockDim.x) K->profA[t] = (uint8_t)bsx_profile_a(A.s, A.I, t >> 4, t & 15);
    #pragma unroll 1
    for (int t = threadIdx.x; t < 160; t += blockDim.x) { K->segof[t] = (uint8_t)(t / A.s); K->remof[t] = (uint8_t)(t % A.s); }
    // chr_lut[g] = largest k with anchor[k] <= g << 24 (0 when none): int2hit then searches [chr_lut[g], chr_lut[g+1]]
    #pragma unroll 1
    for (int t = threadIdx.x; t < 258; t += blockDim.x) {
        int left = 0;
        if (t < 256 && A.n_seq < 65536u) {
            const uint32_t x = (uint32_t)t << 24;
            int right = (int)A.n_seq;
            while (left < right - 1) { const int mid = (left + right) / 2; if (x >= A.seqinfo[mid]) left = mid; else right = mid; }
        } else if (A.n_seq < 65536u) left = (int)A.n_seq - 1;
        K->chr_lut[t] = (uint16_t)left;
    }
    __syncthreads();
}

// A prepared image (bsx_prep.cuh) -> this warp's shared memory: one or two coalesced loads per lane, then the per-read
// state and the context flanks (the read bases that face an entry's inline context, one plan entry per lane).
// ld.cg: the image was written by another lane of this warp moments ago, so the read-only path is not allowed.
__device__ __forceinline__ void load_image(const MapArgs &A, ReadSm *R, const uint8_t *img, int lane) {
    __syncwarp();
    const uint4 hd = __ldcg(reinterpret_cast<const uint4 *>(img));
    const int len = (int)(hd.y & 0xffu), rmsn = (int)((hd.y >> 8) & 0xffu), seg = (int)((hd.y >> 16) & 0xffu);
    const int filtered = (int)((hd.y >> 24) & 1u), fc = (int)((hd.y >> 25) & 1u), cc = (int)((hd.y >> 26) & 1u);
    const int per = MapKernel::rrbs ? 1 : A.I, used = seg * per;
    if (!filtered) {
        #pragma unroll 1
        for (int c = 0; c < A.nslot; c++) {
            const int chain = A.nslot == 2 ? c : (fc ? 0 : 1);
            const uint8_t *sp = img + sizeof(ImgHdr) + (size_t)c * A.img_slot;
            if (lane < 2 * BSX_FIXWORDS) {
                const uint32_t v = __ldcg(reinterpret_cast<const uint32_t *>(sp) + lane);
                if (lane < BSX_FIXWORDS) R->rw[chain][lane] = v; else R->m5[chain][lane - BSX_FIXWORDS] = v;
            }
            uint4 *pl = plan_of(R, chain, A);
            const uint4 *src = reinterpret_cast<const uint4 *>(sp + 2 * BSX_FIXWORDS * 4);
            #pragma unroll 1
            for (int t = lane; t < used; t += 32) pl[t] = __ldcg(src + t);
        }
    }
    if (lane < 16) reinterpret_cast<uint32_t *>(R->nh)[lane] = 0u;      // nh[16], nc[16]
    if (lane == 0) {
        R->raw = (int)(hd.z & 0xffu); R->readset = (int)((hd.z >> 8) & 0xffu); R->seedseg = seg; R->filtered = filtered;
        R->index = hd.x; R->len = len; R->rmsn = rmsn; R->nw = (len + 15) >> 4;
        R->thres = (uint32_t)rmsn; R->fc = fc; R->cc = cc; R->dn = 0; R->best = 99;
    }
    __syncwarp();
    if (!filtered) {
        #pragma unroll 1
        for (int c = 0; c < A.nslot; c++) {
            const int chain = A.nslot == 2 ? c : (fc ? 0 : 1);
            const uint4 *pl = plan_of(R, chain, A);
            uint4 *fl = flank_of(R, chain, A);
            #pragma unroll 1
            for (int t = lane; t < used; t += 32) {
                const int p = (int)(pl[t].w & 0xffffu);
                const uint2 wb = read_window(R, chain, p - 16), wa = read_window(R, chain, p + A.s);
                fl[t * FW] = make_uint4(wb.x, flank_mask(wb.x, wb.y), wa.x, flank_mask(wa.x, wa.y));
                if constexpr (MapKernel::wide) {
                    const uint2 wb2 = read_window(R, chain, p - 32), wa2 = read_window(R, chain, p + A.s + 16);
                    fl[t * FW + 1] = make_uint4(wb2.x, flank_mask(wb2.x, wb2.y), wa2.x, flank_mask(wa2.x, wa2.y));
                }
            }
        }
    }
    __syncwarp();
}

// Phase A for a block of `cnt` units starting at unit u0: lane i prepares unit u0 + i into image i of the warp's scratch
__device__ __forceinline__ void prepare_block(const MapArgs &A, const CtaSm *K, PrepCol *P, uint8_t *scratch, uint32_t u0, uint32_t cnt, int lane, Ctr *C) {
    int np = 0;
    if ((uint32_t)lane < cnt) np = bsx_prep_unit(A, K, &P->rw[0][lane], &P->m5[0][lane], u0 + (uint32_t)lane, scratch + (size_t)lane * A.img_bytes);
#pragma unroll
    for (int d = 16; d; d >>= 1) np += __shfl_xor_sync(BSX_FULL, np, d);
    CTR_ADD(C, CT_PROBE, np);
    __syncwarp();
}

// ------------------------------------------------------------------ K4: extension
// which 16-byte chunk of the window to gather first: for every residue o = (word index & 3) pick
// delta in {0,1,2} maximising the number of valid read bases outside the seed that the chunk's
// three fully covered read words hold.  Returns delta for o = 0..3 packed 2 bits each.
__device__ __forceinline__ uint32_t chunk_table(const ReadSm *R, int chain, int nw, int zlo, int zhi, int lane) {
    const int o = (lane / 3) & 3, dl = lane % 3;
    int score = 0;
    if (lane < 12) {
        const int jlo = 4 * dl - o;
#pragma unroll
        for (int t = 0; t < 3; t++) {
            const int j = jlo + t;
            if (j >= 0 && j < nw) {
                int lo = max(zlo, 16 * j) - 16 * j, hi = min(zhi, 16 * j + 16) - 16 * j;
                uint32_t seedm = 0;
                if (lo < hi) {
                    uint32_t a = 0xffffffffu >> (2 * lo);
                    uint32_t b = (hi >= 16) ? 0u : (0xffffffffu >> (2 * hi));
                    seedm = a & ~b;
                }
                score += __popc(R->m5[chain][j] & ~seedm);
            }
        }
    }
    const int oo = lane & 3;
    const int a0 = __shfl_sync(BSX_FULL, score, 3 * oo), a1 = __shfl_sync(BSX_FULL, score, 3 * oo + 1),
              a2 = __shfl_sync(BSX_FULL, score, 3 * oo + 2);
    int best = 0, bs = a0;
    if (a1 > bs) { best = 1; bs = a1; }
    if (a2 > bs) { best = 2; }
    uint32_t tb = (uint32_t)best << (2 * oo);
    return __shfl_sync(BSX_FULL, tb, 0) | __shfl_sync(BSX_FULL, tb, 1) | __shfl_sync(BSX_FULL, tb, 2) | __shfl_sync(BSX_FULL, tb, 3);
}

__device__ __forceinline__ uint32_t partial_mismatch(const ReadSm *R, int chain, int nw, const uint32_t *__restrict__ refbase,
                                                     uint32_t loc, uint32_t tbl) {
    const uint32_t wi = loc >> 4, sh2 = (loc & 15u) * 2u, o = wi & 3u;
    const uint32_t dl = (tbl >> (2 * o)) & 3u;
    const int jlo = 4 * (int)dl - (int)o;
    // ld.global.nc with a 64-byte L2 fetch: the default promotes every miss to a full 128-byte line
    // (measured: 121 B of HBM traffic per 16-byte gather vs 62 B with .L2::64B, profiles/ubench)
    uint4 c;
    {
        const uint4 *gp = reinterpret_cast<const uint4 *>(refbase) + (wi >> 2) + dl;
        asm volatile("ld.global.nc.L2::64B.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(c.x), "=r"(c.y), "=r"(c.z), "=r"(c.w) : "l"(gp));
    }
    uint32_t w = 0;
    int j = jlo;
    if (j >= 0 && j < nw) w += __popc(bsx_mm_word_bits(R->rw[chain][j], R->m5[chain][j], __funnelshift_l(c.y, c.x, sh2)));
    j++;
    if (j >= 0 && j < nw) w += __popc(bsx_mm_word_bits(R->rw[chain][j], R->m5[chain][j], __funnelshift_l(c.z, c.y, sh2)));
    j++;
    if (j >= 0 && j < nw) w += __popc(bsx_mm_word_bits(R->rw[chain][j], R->m5[chain][j], __funnelshift_l(c.w, c.z, sh2)));
    return w;
}

// CountMismatch (align.h:167-200) over the whole read; stops early once above the threshold
// (measured: requesting all window words up front is 10 % slower on config 2 -- most phase-1 survivors
// are rejected within the first two words)
__device__ __forceinline__ uint32_t full_mismatch(const ReadSm *R, int chain, int nw, const uint32_t *__restrict__ refbase,
                                                  uint32_t loc, uint32_t thres) {
    const uint32_t *rp = refbase + (loc >> 4);
    const uint32_t sh2 = (loc & 15u) * 2u;
    uint32_t w = 0, prev = __ldg(rp);
    #pragma unroll 1
    for (int j = 0; j < nw; j++) {
        const uint32_t next = __ldg(rp + j + 1);
        w += __popc(bsx_mm_word_bits(R->rw[chain][j], R->m5[chain][j], __funnelshift_l(next, prev, sh2)));
        prev = next;
        if (w > thres) break;
    }
    return w;
}

// RefSeq::CCGG_seglen (dbseq.cpp:541-567), clamped at the last site (App. B Q20)
__device__ int ccgg_seglen(const MapArgs &A, uint32_t chr, uint32_t pos, int readlen) {
    const uint32_t *st = A.sites + A.site_off[chr >> 1];
    const int n = (int)(A.site_off[(chr >> 1) + 1] - A.site_off[chr >> 1]);
    int left = 0, right = n - 1;
    while (left < right - 1) {
        int mid = (left + right) / 2;
        uint32_t mv = st[mid];
        if (mv == pos) { left = mid; right = mid + 1; break; }
        else if (mv < pos) left = mid; else right = mid;
    }
    const uint32_t seg_start = st[left], add = (uint32_t)(A.site_len - 2 * A.digest_pos);
    uint32_t seg_end;
    for (;;) {
        int rr = right < n ? right : n - 1;
        seg_end = st[rr] + add;
        if (seg_end < pos + (uint32_t)readlen && right < n) right++; else break;
    }
    return (int)(seg_end - seg_start);
}

// One accepted candidate, executed warp-uniformly: int2hit, bounds, dedupe, bucket append, exits
// (align.cpp:270-278 and its three twins).  Returns 1 when SnpAlign must return.
__device__ int commit_hit(const MapArgs &A, ReadSm *R, uint2 *hits, uint32_t *dd, int store_all, int chain,
                          uint32_t chr, uint32_t loc, uint32_t w, int mode, int frag_filter, int lane, Ctr *C) {
    const uint32_t *anchor = A.seqinfo, *size = A.seqinfo + A.n_seq + 1, *rcoff = A.seqinfo + 2 * A.n_seq + 1;
    const uint32_t k = chr >> 1;
    if (chr & 1u) loc = rcoff[k] - (uint32_t)R->len - loc;
    if (loc + (uint32_t)R->len > size[k]) return 0;                      // overflow the end of refseq
    const uint32_t key = anchor[k] + loc;                               // == (chr>>1, loc), see DESIGN.md
    bool found = false;
    const uint32_t dn = R->dn;
    #pragma unroll 1
    for (uint32_t t = lane; t < dn; t += 32) found |= (dd[t] == key);
    if (__any_sync(BSX_FULL, found)) return 0;                          // hit already exists
    if (dn < A.dd_stride) {                                              // capacity guard (RRBS fragment-filtered hits are uncounted)
        __syncwarp();
        if (lane == 0) { dd[dn] = key; R->dn = dn + 1; }
        __syncwarp();
    }
    if (frag_filter) {
        const int sl = ccgg_seglen(A, chr, loc, R->len);
        if (sl > A.max_insert || sl < A.min_insert) { __syncwarp(); return 0; }
    }
    if ((int)w < R->best) WSET(R->best, (int)w);       // lowest level that holds a hit
    if (lane == 0) {                                    // the bucket counters are lane 0's: nobody else reads them before the fence
        const uint32_t cnt = chain ? R->nc[w] : R->nh[w];
        if (store_all) hits[((size_t)w * 2 + chain) * (A.W + 1) + cnt] = make_uint2(chr, loc);
        else if ((int)w == R->best) hits[(size_t)chain * (A.W + 1) + cnt] = make_uint2(chr, loc);
        if (chain) R->nc[w] = (uint16_t)(cnt + 1); else R->nh[w] = (uint16_t)(cnt + 1);
    }
    __syncwarp();
    CTR_ADD(C, CT_COMMIT, 1);
    const int tot = (int)R->nh[w] + (int)R->nc[w];
    if ((int)w == mode && !A.pairend && A.r == 0 && tot > 1) return 1;
    if (tot >= A.W) { if (w == 0) return 1; WSET(R->thres, w - 1); }
    return 0;
}

// 32 candidates that survived phase 0 (table entries idx0 + lane of one list): phase 1 (one aligned 16-byte
// gather), phase 2 (whole window, exact CountMismatch) and the ordered commit.  Everything a survivor
// needs is re-derived here from its table index, so the filter loop carries no state for it.
// Returns 1 when SnpAlign must return; `last` = exiting lane.
__device__ __forceinline__ int extend_and_commit(const MapArgs &A, ReadSm *R, uint2 *hits, uint32_t *dd,
                                              int store_all, int chain, int mode, bool pass, uint32_t idx0, uint32_t md,
                                              uint32_t p, uint32_t tbl, int use_p1, int lane, Ctr *C) {
    const uint32_t *anchor = A.seqinfo;
    uint32_t strand = 0, loc = anchor[0], chr = 0;
    if (pass) {
        const uint32_t idx = idx0 + lane;
        uint32_t entry;                                                   // a random 4-byte read: 64-byte HBM fetch
        asm volatile("ld.global.nc.L2::64B.u32 %0, [%1];" : "=r"(entry) : "l"(A.pos + idx));
        if constexpr (!MapKernel::rrbs) { strand = idx >= md; loc = entry - p; }           // h = -profile.a + i - seed_start_array
        else {
            chr = __ldg(A.tag + idx) & 0xffffu; strand = chr & 1u; loc = entry - p + anchor[chr >> 1];
            if (entry < p) pass = false;                                      // underflow the start of refseq (align.cpp:194, 236)
        }
    }
    const uint32_t *refbase = strand ? A.crefcat : A.refcat;
    uint32_t w = 0xffffu;
    if (use_p1) {                                                        // many survivors: one 16-byte gather filters first
        CTR_ADD(C, CT_GATHER, __popc(__ballot_sync(BSX_FULL, pass)));
        if (pass) {
            w = partial_mismatch(R, chain, R->nw, refbase, loc, tbl);
            pass = w <= R->thres;
        }
    }
    const unsigned pm1 = __ballot_sync(BSX_FULL, pass);
    unsigned pm = 0;
    if (pm1) {
        if (__popc(pm1) <= 4) {
            // few survivors (the usual case, up to four): the warp counts them two at a time, lanes 16g + j taking word j of
            // survivor g -- one memory round trip per pair instead of a serial walk over the window per lane
            const int nw = R->nw, j = lane & 15, g = lane >> 4;
            unsigned left = pm1;
            #pragma unroll 1
            while (left) {
                const int s0 = __ffs(left) - 1; left &= left - 1;
                const int s1 = left ? __ffs(left) - 1 : -1; if (left) left &= left - 1;
                const int src = g ? s1 : s0;
                const uint32_t loc_g = __shfl_sync(BSX_FULL, loc, src < 0 ? 0 : src);
                const uint32_t strand_g = __shfl_sync(BSX_FULL, strand, src < 0 ? 0 : src);
                uint32_t wj = 0;
                if (src >= 0 && j < nw) {
                    const uint32_t *rp = (strand_g ? A.crefcat : A.refcat) + (loc_g >> 4) + j;
                    const uint32_t a = __ldg(rp), b = __ldg(rp + 1);
                    wj = __popc(bsx_mm_word_bits(R->rw[chain][j], R->m5[chain][j], __funnelshift_l(b, a, (loc_g & 15u) * 2u)));
                }
#pragma unroll
                for (int d = 8; d; d >>= 1) wj += __shfl_xor_sync(BSX_FULL, wj, d);
                const uint32_t w0 = __shfl_sync(BSX_FULL, wj, 0), w1 = __shfl_sync(BSX_FULL, wj, 16);
                if (lane == s0) w = w0;
                if (lane == s1) w = w1;
            }
            if (pass) pass = w <= R->thres;
        } else if (pass) {
            w = full_mismatch(R, chain, R->nw, refbase, loc, R->thres);
            pass = w <= R->thres;
        }
        pm = __ballot_sync(BSX_FULL, pass);
        CTR_ADD(C, CT_FULL, __popc(pm1));
    }
    int ret = 0, last = 31;
    while (pm) {
        const int src = __ffs(pm) - 1;
        pm &= pm - 1;
        const uint32_t w_s = __shfl_sync(BSX_FULL, w, src);
        if (w_s > R->thres) continue;                                     // threshold lowered by an earlier commit
        uint32_t loc_s = __shfl_sync(BSX_FULL, loc, src);
        const uint32_t strand_s = __shfl_sync(BSX_FULL, strand, src);
        uint32_t chr_s;
        if constexpr (!MapKernel::rrbs) {
            // RefSeq::int2hit (dbseq.cpp:585-595); the per-CTA table narrows the search to the sequences
            // that overlap the position's 16 Mb granule (almost always one)
            int left = 0, right = (int)A.n_seq;
            if (A.n_seq < 65536u) { const CtaSm *K = cta_tables(); left = K->chr_lut[loc_s >> 24]; right = K->chr_lut[(loc_s >> 24) + 1] + 1; }
            while (left < right - 1) { int mid = (left + right) / 2; if (loc_s >= anchor[mid]) left = mid; else right = mid; }
            chr_s = (uint32_t)left * 2u + strand_s;
            loc_s -= anchor[left];
        } else {
            chr_s = __shfl_sync(BSX_FULL, chr, src);
            loc_s -= anchor[chr_s >> 1];
        }
        ret = commit_hit(A, R,  hits, dd, store_all, chain, chr_s, loc_s, w_s, mode,
                         MapKernel::rrbs && chain == 0 && !A.pairend, lane, C);
        if (ret) { last = src; break; }
    }
    return ret | (last << 8);        // bit 0: SnpAlign returns; bits 8..: exiting lane
}

// Per-warp staging area of the packed list walk; aliases the prepare phase's PrepCol (idle while the warp aligns).
// A context entry is {16 bases before the seed, 16 after it}; wide: {bases -32..-17, -16..-1 before, +0..+15, +16..+31 after}.
// A half-step is 32 consecutive entries of one position list.
struct NarrowStep {
    uint4 d;                            // first entry index, list start, list length (0: padding), list number within the mode
    uint4 f;                            // the read bases / flank_mask that face the list's inline context before / after the seed
};
struct WideStep {
    uint4 d, f;
    uint4 f2;                           // the same for the outer 16 + 16 bases
};
typedef std::conditional_t<MapKernel::wide, uint4, uint2> CtxEntry;
typedef std::conditional_t<MapKernel::wide, WideStep, NarrowStep> HalfStep;
struct StageSm {
    CtxEntry slot[ROUND_HS * 32];       // one round of ROUND_HS half-steps x 32 entries
    HalfStep sched[ROUND_HS];
};
// the staging area aliases the idle PrepCol plus bsx_stage_extra_bytes() behind it (bsx_warp_smem_bytes)
static_assert(ROUND_HS % 2 == 0 && ROUND_HS <= 32, "half-steps are evaluated in pairs; one lane describes one half-step");

// mismatches among the read bases that face one entry's inline context (flanks f of its half-step): a lower bound of
// CountMismatch
__device__ __forceinline__ uint32_t ctx_count(const NarrowStep &h, const uint2 c) { return ctx_mm2(h.f, c); }
__device__ __forceinline__ uint32_t ctx_count(const WideStep &h, const uint4 c) {
    return ctx_mm2(h.f, make_uint2(c.y, c.z)) + ctx_mm2(h.f2, make_uint2(c.x, c.w));
}

// SnpAlign returned at lane `xl` of half-step `cur` of the current round: the candidates the sequential reference has
// visited are the lists before this one and this list up to the exiting entry; everything else that was requested
// in this round is over-fetch, the rounds that were never requested do not count at all.
__device__ __noinline__ void packed_exit(const uint4 *plan, int per, StageSm *S, uint32_t cur, uint32_t xl, int lane, Ctr *C) {
    const uint4 sc = S->sched[cur].d;
    uint32_t nk = 0;
    if (lane < per) { const uint4 el = plan[lane]; nk = el.z - el.x; }
    const uint32_t all = __reduce_add_sync(BSX_FULL, nk);
    const uint32_t before = __reduce_add_sync(BSX_FULL, (uint32_t)lane < sc.w ? nk : 0u);
    const uint32_t counted = before + (sc.x + xl - sc.y) + 1u;
    uint32_t extra = 0;                                                   // entries of this round behind the exiting one
    if (lane < ROUND_HS && (uint32_t)lane >= cur) {
        const uint4 t = S->sched[lane].d;
        uint32_t lo_i = max(t.x, t.y);
        const uint32_t hi_i = min(t.x + 32u, t.y + t.z);
        if ((uint32_t)lane == cur) lo_i = max(lo_i, t.x + xl + 1u);
        extra = hi_i > lo_i ? hi_i - lo_i : 0u;
    }
    const uint32_t req = counted + __reduce_add_sync(BSX_FULL, extra);
    if (lane == 0) { C[CT_LIST] -= all - req; C[CT_OVER] += req - counted; }
}

// phase-1 chunk choice for a mode: keep away from its seed zone (all sub-seeds)
__device__ __noinline__ uint32_t mode_chunk_table(const MapArgs &A, const ReadSm *R, int chain, const uint4 *plan, int per, int lane) {
    int zlo = 1000, zhi = -1;
    if (lane < per) { zlo = zhi = (int)(plan[lane].w & 0xffffu); }
#pragma unroll
    for (int d = 8; d; d >>= 1) { zlo = min(zlo, __shfl_xor_sync(BSX_FULL, zlo, d)); zhi = max(zhi, __shfl_xor_sync(BSX_FULL, zhi, d)); }
    zlo = __shfl_sync(BSX_FULL, zlo, 0); zhi = __shfl_sync(BSX_FULL, zhi, 0) + A.s;
    return chunk_table(R, chain, R->nw, zlo, zhi, lane);
}

// SnpAlign for one mode (align.cpp:168-347), lists staged through shared memory.
// The position lists of the mode (WGBS: its I sub-seeds; RRBS: the one (segment, mirror) group of its key) are cut into
// half-steps of 32 entries -- a list starts a new half-step (8-byte entries: at the even entry index at or before its
// first entry, so that every copy is a 16-byte cp.async) -- and the half-steps of all lists form one schedule that is
// fetched in rounds of ROUND_HS and evaluated two half-steps = 64 candidates at a time: one DRAM round trip per round
// instead of one per list.  Indexes built for -v >= 8 carry 16-byte entries (32 + 32 context bases): 32 bases let a fifth
// of config 5's candidates through; the first design kept the outer bases in a second array read by survivors only,
// which cost one dependent random access per 64-candidate step.  Lane t of the warp describes half-step t of the round (which list, where it starts, the read bases that face
// its context); within a half-step the list is warp-uniform, so a candidate costs one 8-byte shared-memory load, eight
// logic operations, one popcount and a compare.  The fast path does not even test whether a staged entry belongs to
// the list: stale or foreign entries can only raise a false alarm, which the slow path masks out.  Candidates are
// visited in the reference's order, so commits, -w threshold lowering and the early returns fire exactly where the
// sequential reference stops.  (A template only so that `if constexpr` drops the wide half-step's members from the
// other kernels.)
template <class Step = HalfStep>
__device__ __forceinline__ int snp_align_packed(const MapArgs &A, ReadSm *R, uint2 *hits, uint32_t *dd, int store_all, int mode, int lane, Ctr *C, StageSm *S) {
    const int per = MapKernel::rrbs ? 1 : A.I;
    const int chain_lo = R->fc ? 0 : 1, chain_hi = R->cc ? 2 : 1;          // the chains this read is searched on (fixed per read)
    #pragma unroll 1
    for (int chain = chain_lo; chain < chain_hi; chain++) {
        const uint4 *plan = plan_of(R, chain, A) + mode * per, *flank = flank_of(R, chain, A) + mode * per * FW;
        uint4 e = make_uint4(0u, 0u, 0u, 0u);                             // lane k < per owns list k: {start, rc start, end, p | segment << 16}
        if (lane < per) e = plan[lane];
        const uint32_t n = e.z - e.x;
        uint32_t cum = n ? (n + (MapKernel::wide ? 0u : (e.x & 1u)) + 31u) >> 5 : 0u;   // half-steps of my list -> inclusive scan over the lists
        const uint32_t my_hs = cum;
        #pragma unroll 1
        for (int d = 1; d < per; d <<= 1) { const uint32_t t = __shfl_up_sync(BSX_FULL, cum, d); if (lane >= d) cum += t; }
        const uint32_t total_hs = __shfl_sync(BSX_FULL, cum, per - 1);
        if (total_hs == 0) continue;
        CTR_ADD(C, CT_LIST, __reduce_add_sync(BSX_FULL, n));              // corrected by packed_exit when SnpAlign returns early
        uint32_t thres = R->thres;
        uint32_t run_end = 0;                                             // run_advance: running total of the list the previous round ended in
        #pragma unroll 1
        for (uint32_t h0 = 0; h0 < total_hs; h0 += ROUND_HS) {
            if (MapKernel::run_advance && h0 + ROUND_HS <= run_end) {
                // a long list: every half-step of this round continues the list the previous round ended in, so the
                // schedule is that round's last entry moved on by 32 entries per half-step
                Step h = S->sched[ROUND_HS - 1];
                __syncwarp();
                if (lane < ROUND_HS) { h.d.x += 32u * ((uint32_t)lane + 1u); S->sched[lane] = h; }
                __syncwarp();
            } else if constexpr (MapKernel::owner_sched) {
                // the lane that owns list j writes the descriptors of the list's half-steps that fall into this round; the
                // tail of the round (past the mode's last half-step) is padding: no entry of it is ever inside a list
                const uint32_t first = cum - my_hs;                       // my list's first half-step in the mode's sequence
                if constexpr (MapKernel::run_advance) {                   // where the list of this round's last half-step ends
                    const uint32_t idx = h0 + ROUND_HS - 1u;
                    const unsigned own = __ballot_sync(BSX_FULL, lane < per && first <= idx && idx < cum);
                    const uint32_t ce = __shfl_sync(BSX_FULL, cum, own ? __ffs(own) - 1 : 0);
                    run_end = own ? ce : 0u;
                }
                __syncwarp();                                             // the previous round's slow path may still read the schedule
                if (lane < ROUND_HS && h0 + (uint32_t)lane >= total_hs) S->sched[lane] = Step{};
                if (lane < per && my_hs) {
                    const uint32_t lo = max(first, h0), hi = min(cum, h0 + (uint32_t)ROUND_HS);
                    if (lo < hi) {
                        Step h;
                        h.f = flank[lane * FW];
                        if constexpr (MapKernel::wide) h.f2 = flank[lane * FW + 1];
                        h.d = make_uint4((MapKernel::wide ? e.x : (e.x & ~1u)) + 32u * (lo - first), e.x, n, (uint32_t)lane);
                        #pragma unroll 1
                        for (uint32_t t = lo; t < hi; t++) { S->sched[t - h0] = h; h.d.x += 32u; }
                    }
                }
                __syncwarp();
            } else {
                // lane t describes half-step h0 + t: its list is the first one whose running total exceeds h0 + t.  One
                // shuffle per list, independent of each other (a binary search over the lanes that hold the totals
                // measured -9 % on paired-end: a dependent chain; the loop unrolled x4 lost too)
                const uint32_t target = h0 + (uint32_t)lane;
                int k = 0; uint32_t first = 0;
                #pragma unroll 1
                for (int j = 0; j < per; j++) { const uint32_t c = __shfl_sync(BSX_FULL, cum, j); if (c <= target) { k = j + 1; first = c; } }
                if constexpr (MapKernel::run_advance) {                   // where the list of this round's last half-step ends
                    const int kk = __shfl_sync(BSX_FULL, k, ROUND_HS - 1);
                    const uint32_t ce = __shfl_sync(BSX_FULL, cum, kk & 15);
                    run_end = kk < per ? ce : 0u;
                }
                __syncwarp();                                             // the previous round's slow path may still read the schedule
                if (lane < ROUND_HS) {
                    Step h{};                                             // padding: no entry of it is ever inside a list
                    if (k < per) {
                        const uint4 ek = plan[k];
                        h.d = make_uint4((MapKernel::wide ? ek.x : (ek.x & ~1u)) + 32u * (target - first), ek.x, ek.z - ek.x, (uint32_t)k);
                        h.f = flank[k * FW];
                        if constexpr (MapKernel::wide) h.f2 = flank[k * FW + 1];
                    }
                    S->sched[lane] = h;
                }
                __syncwarp();
            }
            if constexpr (MapKernel::wide) {
                // 16-byte entries: lane L stages entry L of every half-step of the round (512 contiguous bytes per copy)
                const char *ctx = reinterpret_cast<const char *>(A.ctx) + 16u * (uint32_t)lane;
                uint32_t sp = (uint32_t)__cvta_generic_to_shared(&S->slot[lane]);
                asm volatile("" : "+r"(sp), "+l"(ctx));                   // opaque: computed once, not rematerialised under each predicate
#pragma unroll
                for (uint32_t q = 0; q < ROUND_HS; q++) {
                    const uint4 sc = S->sched[q].d;
                    if (sc.x + (uint32_t)lane < sc.y + sc.z) cp_async16s(sp + 512u * q, ctx + (size_t)sc.x * 16u);
                }
            } else {
                // sixteen lanes stage one half-step: 256 contiguous bytes per half-warp and copy (four lanes per half-step
                // measured slower)
                const uint32_t half = (uint32_t)lane >> 4, pr = 2u * ((uint32_t)lane & 15u);
                const char *ctx = reinterpret_cast<const char *>(A.ctx) + 8u * pr;
                uint32_t sp = (uint32_t)__cvta_generic_to_shared(&S->slot[half * 32u + pr]);
                asm volatile("" : "+r"(sp), "+l"(ctx));                   // opaque: computed once, not rematerialised under each predicate
#pragma unroll
                for (uint32_t q = 0; q < ROUND_HS / 2; q++) {
                    const uint4 sc = S->sched[2u * q + half].d;
                    if (sc.x + pr < sc.y + sc.z) cp_async16s(sp + 512u * q, ctx + (size_t)sc.x * 8u);
                }
            }
            cp_async_commit();
            cp_async_wait<0>();
            __syncwarp();
            const uint32_t nst = min((uint32_t)ROUND_HS, total_hs - h0);
            #pragma unroll 1
            for (uint32_t hs = 0; hs < nst; hs += 2) {
                bool pass0 = ctx_count(S->sched[hs], S->slot[hs * 32u + lane]) <= thres;
                bool pass1 = ctx_count(S->sched[hs + 1], S->slot[hs * 32u + 32u + lane]) <= thres;
                if (!__any_sync(BSX_FULL, pass0 || pass1)) continue;
                // ---- slow path: some staged entry passed the inline-context filter; is it a candidate at all?
                const uint4 s0 = S->sched[hs].d, s1 = S->sched[hs + 1].d;
                pass0 &= (s0.x + (uint32_t)lane - s0.y) < s0.z;                                  // inside the list (unsigned; padding has length 0)
                pass1 &= (s1.x + (uint32_t)lane - s1.y) < s1.z;
                const unsigned pm0 = __ballot_sync(BSX_FULL, pass0), pm1 = __ballot_sync(BSX_FULL, pass1);
                if (!(pm0 | pm1)) continue;
                // phase 1 (one aligned 16-byte gather per survivor) only pays when phase 0 lets many through
                const int use_p1 = __popc(pm0) + __popc(pm1) > 2;
                const uint32_t tbl = use_p1 ? mode_chunk_table(A, R, chain, plan, per, lane) : 0u;
                int ret = 0;
#pragma unroll 1
                for (int h = 0; h < 2; h++) {                            // one call site: the slow path exists once in the binary
                    if (h ? pm1 : pm0) {
                        const uint4 sc = h ? s1 : s0;
                        const uint4 ek = plan[sc.w];
                        const int rc = extend_and_commit(A, R, hits, dd, store_all, chain, mode, h ? pass1 : pass0, sc.x, ek.y, ek.w & 0xffffu, tbl, use_p1, lane, C);
                        if (rc & 1) { packed_exit(plan, per, S, hs + (uint32_t)h, (uint32_t)(rc >> 8), lane, C); ret = 1; break; }
                    }
                }
                if (ret) return 1;
                thres = R->thres;
            }
        }
    }
    return 0;
}

// SingleAlign::RunAlign (align.cpp:435-452): the mode loop (everything before it happened in the prepare kernel)
__device__ __forceinline__ void run_align(const MapArgs &A, ReadSm *R, uint2 *hits, uint32_t *dd, int store_all, int lane, Ctr *C, StageSm *stage) {
    #pragma unroll 1
    for (int m = 0; m < R->seedseg; m++) {
        snp_align_packed(A, R, hits, dd, store_all, m, lane, C, stage);
        if (!MapKernel::rrbs && R->best <= m) return;   // a bucket <= m is non-empty (align.cpp:448)
    }
}

// StringAlign (align.cpp:610-627) -> record
__device__ void write_record(const MapArgs &A, const ReadSm *R, const uint2 *hits, int store_all,
                             bsx_rec *out, uint16_t *cnt, int lane) {
    if (cnt && lane < 16) cnt[lane] = (!R->filtered && lane <= R->rmsn) ? (uint16_t)(R->nh[lane] + R->nc[lane]) : (uint16_t)0;
    if (lane != 0) return;
    bsx_rec o;
    o.loc = 0; o.chr = 0; o.nhits = 0; o.nm = 0; o.chain = 0; o.status = (uint8_t)R->filtered; o.len = (uint8_t)R->len;
    if (!R->filtered) {
        const int ii = R->best <= R->rmsn ? R->best : R->rmsn + 1;     // lowest non-empty bucket
        const int sum = ii <= R->rmsn ? R->nh[ii] + R->nc[ii] : 0;
        o.nm = (uint8_t)ii;
        if (sum > 0) {
            const int j = sum > 1 ? (int)(bsx_myrand(R->index, A.randseed) % (uint32_t)sum) : 0;   // a unique hit needs no draw (and no division)
            const int nh = R->nh[ii];
            const int chain = j >= nh;
            const size_t lvl = store_all ? (size_t)ii * 2 : 0;
            const uint2 h = hits[(lvl + chain) * (A.W + 1) + (chain ? j - nh : j)];
            o.chr = h.x; o.loc = h.y; o.nhits = (uint32_t)sum; o.chain = (uint8_t)chain;
        }
    }
    *out = o;
}

__device__ __forceinline__ void flush_counters(const MapArgs &A, Ctr *C, int lane) {
    __syncwarp();
    // candidates the reference semantics visit = list entries requested - entries evaluated past an exit point
    if (lane < 8) { atomicAdd(A.stats + lane, (unsigned long long)(lane == CT_CAND ? C[CT_LIST] - C[CT_OVER] : C[lane])); }
    __syncwarp();
    if (lane < 8) C[lane] = 0;
    __syncwarp();
}

// ------------------------------------------------------------------ SE kernel
__device__ __forceinline__ void map_se(const MapArgs &A) {
    extern __shared__ __align__(16) uint8_t smem[];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    CtaSm *K = reinterpret_cast<CtaSm *>(smem);
    init_cta_tables(A, K);
    uint8_t *base = smem + sizeof(CtaSm) + A.warp_smem_se * wid;
    ReadSm *R = reinterpret_cast<ReadSm *>(base);
    SelSm *X = reinterpret_cast<SelSm *>(base + A.read_smem);
    PrepCol *P = reinterpret_cast<PrepCol *>(base + A.read_smem + sizeof(SelSm));
    const uint32_t gw = blockIdx.x * (blockDim.x >> 5) + wid;
    uint2 *hits = A.hit_scratch + (size_t)gw * A.hit_stride;
    uint32_t *dd = A.dd_scratch + (size_t)gw * A.dd_stride;
    Ctr *C = X->ctr;
    if (lane < 8) C[lane] = 0;
    __syncwarp();
    uint8_t *scratch = A.prep + (size_t)gw * 32u * A.img_bytes;
    for (;;) {
        uint32_t r0 = 0;                        // one atomic hands this warp up to 32 consecutive reads
        if (lane == 0) r0 = atomicAdd(A.work_counter, A.block_units);
        r0 = __shfl_sync(BSX_FULL, r0, 0);
        if (r0 >= A.n) break;
        const uint32_t cnt = min(A.block_units, A.n - r0);
        prepare_block(A, K, P, scratch, r0, cnt, lane, C);                       // phase A: one lane per read
        #pragma unroll 1
        for (uint32_t i = 0; i < cnt; i++) {                                  // phase B: the warp aligns them one by one
            const uint32_t r = r0 + i;
            if (C[CT_LIST] & 0x80000000u) flush_counters(A, C, lane);
            load_image(A, R, scratch + (size_t)i * A.img_bytes, lane);
            if (!R->filtered) run_align(A, R, hits, dd, 0, lane, C, reinterpret_cast<StageSm *>(P));
            __syncwarp();
            write_record(A, R,  hits, 0, A.out_a + r, A.cnt_a ? A.cnt_a + (size_t)r * 16 : nullptr, lane);
            if (!R->filtered && R->best <= R->rmsn) CTR_ADD(C, CT_MAPPED, 1);
            __syncwarp();
        }
    }
    flush_counters(A, C, lane);
}

// ------------------------------------------------------------------ PE kernel (pairs.cpp)
// pair buckets: pairhits[na+nb][..] as uint4 {a.chr, a.loc, b.chr, b.loc}; insert / chain / na / nb
// in a parallel uint4.  One warp per pair; GetPairs runs on lane 0 (its loops are short and strictly
// ordered), the two mates' SnpAlign calls are the warp-parallel part.
struct PairHitDev { uint32_t a_chr, a_loc, b_chr, b_loc; int32_t insert; uint32_t meta; /* chain | na<<8 | nb<<16 */ uint32_t pad0, pad1; };

__device__ void sort_hits(uint2 *h, int n, int lane) {
    // SortHits4PE (align.cpp:363-368) with HitComp (utilities.cpp:53): ascending (chr, loc).  Bucket
    // elements are distinct (dedupe), so any correct sort agrees with std::sort.  Warp-parallel
    // odd-even transposition in place; buckets are almost always 0-2 entries.
    if (n < 2) return;
    bool dirty = true;
    while (dirty) {
        bool sw = false;
        #pragma unroll 1
        for (int phase = 0; phase < 2; phase++) {
            #pragma unroll 1
            for (int i = phase + 2 * lane; i + 1 < n; i += 64) {
                const uint2 a = h[i], b = h[i + 1];
                if (a.x > b.x || (a.x == b.x && a.y > b.y)) { h[i] = b; h[i + 1] = a; sw = true; }
            }
            __syncwarp();
        }
        dirty = __any_sync(BSX_FULL, sw);
    }
}

// GetPairs (pairs.cpp:34-135), lane 0 only
__device__ int get_pairs(const MapArgs &A, const ReadSm *Ra, const ReadSm *Rb,
                         const uint2 *ha_all, const uint2 *hb_all, PairHitDev *pairs, uint16_t *npairs, int na, int nb) {
    if (na > Ra->rmsn || nb > Rb->rmsn) return 0;
    const size_t W1 = (size_t)A.W + 1;
    uint16_t &cnt = npairs[na + nb];
    PairHitDev *bucket = pairs + (size_t)(na + nb) * W1;
    for (int dir = 0; dir < 2; dir++) {
        const uint2 *ha = ha_all + ((size_t)na * 2 + dir) * W1;           // dir 0: a.hits  x b.chits
        const uint2 *hb = hb_all + ((size_t)nb * 2 + (1 - dir)) * W1;     // dir 1: a.chits x b.hits
        const int cnt_a = dir ? Ra->nc[na] : Ra->nh[na];
        const int cnt_b = dir ? Rb->nh[nb] : Rb->nc[nb];
        uint32_t chra = 0xffffffffu; int bstart = 0, bend = 0;
        #pragma unroll 1
        for (int i = 0; i < cnt_a; i++) {
            const uint2 x = ha[i];
            if (chra != x.x) {
                chra = x.x;
                for (bstart = bend; bstart < cnt_b; bstart++) if (hb[bstart].x >= chra) break;
                for (bend = bstart; bend < cnt_b; bend++) if (hb[bend].x > chra) break;
            }
            #pragma unroll 1
            for (int j = bstart; j < bend; j++) {
                const uint2 y = hb[j];
                const bool a_first = dir ? ((chra & 1u) != 0) : ((chra & 1u) == 0);
                uint32_t seg_start, seg_end;
                if (!a_first) { seg_start = y.y; seg_end = x.y + (uint32_t)Ra->len; }
                else { seg_start = x.y; seg_end = y.y + (uint32_t)Rb->len; }
                const int ins = (int)(seg_end - seg_start);
                if (ins >= A.min_insert && ins <= A.max_insert) {
                    PairHitDev ph;
                    ph.a_chr = x.x; ph.a_loc = x.y; ph.b_chr = y.x; ph.b_loc = y.y; ph.insert = ins;
                    ph.meta = (uint32_t)dir | ((uint32_t)na << 8) | ((uint32_t)nb << 16); ph.pad0 = ph.pad1 = 0;
                    bucket[cnt++] = ph;
                    if ((int)cnt >= A.W) return 1;
                }
            }
        }
    }
    return cnt > 0;
}

// the selection half of StringAlignUnpair (pairs.cpp:244-286) for one mate -> record
__device__ void write_unpaired(const MapArgs &A, const ReadSm *R, const uint2 *hits, bsx_rec *out, uint16_t *cnt, int lane) {
    if (cnt && lane < 16) cnt[lane] = (!R->filtered && lane <= R->rmsn) ? (uint16_t)(R->nh[lane] + R->nc[lane]) : (uint16_t)0;
    if (lane != 0) return;
    bsx_rec o;
    o.loc = 0; o.chr = 0; o.nhits = 0; o.nm = 0; o.chain = 0; o.status = (uint8_t)R->filtered; o.len = (uint8_t)R->len;
    if (!R->filtered) {
        int na, ma = 0, ra = 0;
        for (na = 0; na <= R->rmsn; na++) if ((ma = R->nh[na] + R->nc[na]) > 0) break;
        uint2 h = make_uint2(0, 0);
        if (ma) {
            if (ma > 1) ra = (int)(bsx_myrand(R->index, A.randseed) % (uint32_t)ma);
            const int nh = R->nh[na];
            h = (ra < nh) ? hits[((size_t)na * 2) * (A.W + 1) + ra] : hits[((size_t)na * 2 + 1) * (A.W + 1) + (ra - nh)];
        }
        na %= (R->rmsn + 1);
        o.chr = h.x; o.loc = h.y; o.nhits = (uint32_t)ma; o.nm = (uint8_t)na;
        o.chain = (uint8_t)(ra >= (int)R->nh[na]);
    }
    *out = o;
}

// Fix_Unpaired_Short_Fragment (align.cpp:768-791), lane 0
__device__ void fix_unpaired_short(const MapArgs &A, ReadSm *R, uint2 *hits) {
    if (R->len >= A.min_insert) return;
    const size_t W1 = (size_t)A.W + 1;
    #pragma unroll 1
    for (int ii = 0; ii <= R->rmsn; ii++) {
        for (int pass = 0; pass < 2; pass++) {
            uint2 *h = hits + ((size_t)ii * 2 + pass) * W1;
            int cnt = pass ? R->nc[ii] : R->nh[ii];
            #pragma unroll 1
            for (int j = 0; j < cnt; j++) {
                const int sl = ccgg_seglen(A, h[j].x, h[j].y, R->len);
                if (sl < A.min_insert || sl > A.max_insert) { cnt--; for (int k = j; k < cnt; k++) h[k] = h[k + 1]; j--; }
            }
            if (pass) R->nc[ii] = (uint16_t)cnt; else R->nh[ii] = (uint16_t)cnt;
        }
        if (R->nh[ii] + R->nc[ii] > 0) break;
    }
}

__device__ __forceinline__ void map_pe(const MapArgs &A) {
    extern __shared__ __align__(16) uint8_t smem[];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const size_t read_sm = A.read_smem;
    const size_t per_warp = 2 * read_sm + sizeof(SelSm) + sizeof(PrepCol) + bsx_stage_extra_bytes(MapKernel::wide, 1, MapKernel::rrbs);
    CtaSm *K = reinterpret_cast<CtaSm *>(smem);
    init_cta_tables(A, K);
    uint8_t *base = smem + sizeof(CtaSm) + per_warp * wid;
    ReadSm *Ra = reinterpret_cast<ReadSm *>(base);
    ReadSm *Rb = reinterpret_cast<ReadSm *>(base + read_sm);
    SelSm *X = reinterpret_cast<SelSm *>(base + 2 * read_sm);
    PrepCol *P = reinterpret_cast<PrepCol *>(base + 2 * read_sm + sizeof(SelSm));
    const uint32_t gw = blockIdx.x * (blockDim.x >> 5) + wid;
    uint2 *hits_a = A.hit_scratch + (size_t)gw * 2 * A.hit_stride, *hits_b = hits_a + A.hit_stride;
    uint32_t *dd_a = A.dd_scratch + (size_t)gw * 2 * A.dd_stride;                       // mate b: + dd_stride
    PairHitDev *pairs = reinterpret_cast<PairHitDev *>(A.pair_scratch + (size_t)gw * A.pair_stride);
    uint16_t *npairs = X->npairs;
    Ctr *C = X->ctr;
    if (lane < 8) C[lane] = 0;
    __syncwarp();
    const size_t W1 = (size_t)A.W + 1;
    uint8_t *scratch = A.prep + (size_t)gw * 32u * A.img_bytes;
    for (;;) {
        uint32_t r0 = 0;                        // one atomic hands this warp up to 16 consecutive pairs = 32 units
        if (lane == 0) r0 = atomicAdd(A.work_counter, A.block_units >> 1);
        r0 = __shfl_sync(BSX_FULL, r0, 0);
        if (r0 >= A.n) break;
        const uint32_t cnt = min(A.block_units >> 1, A.n - r0);
        prepare_block(A, K, P, scratch, r0 * 2u, cnt * 2u, lane, C);             // phase A: one lane per mate
      #pragma unroll 1
      for (uint32_t pi = 0; pi < cnt; pi++) {                                 // phase B: the warp aligns the pairs one by one
        const uint32_t r = r0 + pi;
        if (C[CT_LIST] & 0x80000000u) flush_counters(A, C, lane);
        // every big device function has exactly one call site (loops over the mate instead of two calls), so the
        // kernel can be inlined whole without holding several copies of the list walk: instruction fetch was the top
        // stall of the version that called them as functions
        #pragma unroll 1
        for (uint32_t mate = 0; mate < 2; mate++)
            load_image(A, reinterpret_cast<ReadSm *>(base + mate * read_sm), scratch + (size_t)(2u * pi + mate) * A.img_bytes, lane);
        int paired = 0;
        bsx_pair_rec po;
        po.a_loc = po.a_chr = po.b_loc = po.b_chr = 0; po.insert = 0; po.npairs = 0; po.na = po.nb = po.chain = po.paired = 0;
        const bool both = !Ra->filtered && !Rb->filtered;
        // both mates usable: PairAlign::RunAlign (pairs.cpp:137-190), level by level until a level pairs.  Otherwise the
        // usable mate runs SingleAlign::RunAlign (align.cpp:435-452): its modes in turn, stopping at the first mode m
        // that leaves a hit at level <= m
        const int maxi = both ? max(Ra->rmsn, Rb->rmsn) : max(Ra->filtered ? -1 : Ra->seedseg - 1, Rb->filtered ? -1 : Rb->seedseg - 1);
        uint32_t done = (Ra->filtered ? 1u : 0u) | (Rb->filtered ? 2u : 0u);      // mates that take no further SnpAlign call
        if (lane < 31) npairs[lane] = 0;
        __syncwarp();
        #pragma unroll 1
        for (int i = 0; i <= maxi && !paired; i++) {
            #pragma unroll 1
            for (uint32_t mate = 0; mate < 2; mate++) {
                if ((done >> mate) & 1u) continue;
                ReadSm *R = reinterpret_cast<ReadSm *>(base + mate * read_sm);
                if (i < R->seedseg) {
                    snp_align_packed(A, R, hits_a + mate * A.hit_stride, dd_a + mate * A.dd_stride, 1, i, lane, C, reinterpret_cast<StageSm *>(P));
                    if (!both && !MapKernel::rrbs && R->best <= i) done |= 1u << mate;   // a bucket <= i is non-empty (align.cpp:448)
                }
            }
            if (!both) continue;
            #pragma unroll 1
            for (uint32_t q = 0; q < 4; q++) {                               // SortHits4PE: level i of both mates, both chains
                const ReadSm *R = reinterpret_cast<const ReadSm *>(base + (q >> 1) * read_sm);
                if (i <= R->rmsn) sort_hits(hits_a + (q >> 1) * A.hit_stride + ((size_t)i * 2 + (q & 1u)) * W1, (q & 1u) ? R->nc[i] : R->nh[i], lane);
            }
            __syncwarp();
            int n = 0;
            if (lane == 0) {
                #pragma unroll 1
                for (int t = 0; t <= 2 * i; t++) {                           // (i,i), then (i,j), (j,i) for j < i
                    const int j = (t - 1) >> 1;
                    n += get_pairs(A, Ra, Rb, hits_a, hits_b, pairs, npairs, (t == 0 || (t & 1)) ? i : j, (t == 0 || !(t & 1)) ? i : j);
                }
            }
            n = __shfl_sync(BSX_FULL, n, 0);
            if (n > 0) paired = i + 1;
        }
        __syncwarp();
        if (paired && lane == 0) {
            // StringAlignPair (pairs.cpp:222-242)
            #pragma unroll 1
            for (int i = 0; i <= A.v * 2; i++) {
                const int np = npairs[i];
                if (!np) continue;
                int j = -1;
                if (np == 1) j = 0;
                else if (A.r == 1) j = (int)(bsx_myrand(Ra->index, A.randseed) % (uint32_t)np);
                if (j >= 0) {
                    const PairHitDev ph = pairs[(size_t)i * W1 + j];
                    po.a_chr = ph.a_chr; po.a_loc = ph.a_loc; po.b_chr = ph.b_chr; po.b_loc = ph.b_loc; po.insert = ph.insert;
                    po.npairs = (uint32_t)np; po.chain = (uint8_t)(ph.meta & 0xff); po.na = (uint8_t)((ph.meta >> 8) & 0xff);
                    po.nb = (uint8_t)((ph.meta >> 16) & 0xff); po.paired = 1;
                }
                break;
            }
        }
        const int out_paired = __shfl_sync(BSX_FULL, (int)po.paired, 0);
        if (lane == 0) A.out_pair[r] = po;
        #pragma unroll 1
        for (uint32_t mate = 0; mate < 2; mate++) {
            ReadSm *R = reinterpret_cast<ReadSm *>(base + mate * read_sm);
            uint2 *hits = hits_a + mate * A.hit_stride;
            if (!out_paired && MapKernel::rrbs) {
                if (lane == 0 && !R->filtered) fix_unpaired_short(A, R, hits);
                __syncwarp();
            }
            uint16_t *cnt16 = mate ? A.cnt_b : A.cnt_a;
            write_unpaired(A, R, hits, (mate ? A.out_b : A.out_a) + r, cnt16 ? cnt16 + (size_t)r * 16 : nullptr, lane);
        }
        if (out_paired) CTR_ADD(C, CT_MAPPED, 1);
        __syncwarp();
      }
    }
    flush_counters(A, C, lane);
}

}  // namespace
