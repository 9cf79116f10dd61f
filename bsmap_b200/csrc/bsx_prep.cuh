// bsx_prep.cuh -- the prepare phase: everything SingleAlign does to a read before the first SnpAlign call,
// one THREAD per read.
//
//   TrimAdapter (align.cpp:371-425) -> FilterReads / CountNs (579-589, 48-55) -> ConvertBinaySeq (90-162)
//   -> seed probing + ReorderSeed / AdjustSeedStartArray / seedindex (454-528, 549-571)
//
// These steps are short, branchy and sequential per read; run by a whole warp (the first design) they cost
// ~1000 warp instructions per read with most lanes idle -- a third of the align kernel, which is issue-bound.
// One thread per read executes the same work in ~1/10 of the warp instructions, because reads of one length
// take identical trip counts and the lanes stay converged.  A warp therefore takes 32 units (reads / mates) at
// a time: phase A, each lane prepares one unit into a compact image (header, packed read, seed plan: bsx_map.cuh)
// in the warp's global scratch; phase B, the warp aligns the 32 units one after the other, expanding each image into
// shared memory (one or two coalesced loads per lane; the context flanks are derived there, one plan entry per lane).  Phase A is latency-bound
// (~30 dependent-free but serial table probes per lane) and hides behind the other warps' phase B.
// (A separate prepare KERNEL was measured first: 209 M reads/s against 268 M -- alone on the GPU it is bound by
// DRAM random accesses, 30 ms per 20 M reads, that the fused form overlaps with issue-bound alignment.)
#pragma once
#include "bsx_map.cuh"

namespace {

typedef CtaSm PrepSm;   // profA / segof / remof live in the CTA's table block

// four ASCII bases in a u32 (first base in the low byte) -> their 2-bit codes and validity, byte-wise
__device__ __forceinline__ void codes4(uint32_t w, uint32_t &code, uint32_t &valid) {
    const uint32_t v = w | 0x20202020u;
    valid = __vcmpeq4(v, 0x61616161u) | __vcmpeq4(v, 0x63636363u) | __vcmpeq4(v, 0x67676767u) | __vcmpeq4(v, 0x74747474u);
    uint32_t c = (w >> 1) & 0x03030303u;          // A 0, C 1, G 3, T 2
    c ^= (c >> 1) & 0x01010101u;                   // A 0, C 1, G 2, T 3
    code = c & valid;                              // everything else -> 0 (alphabet[], param.cpp:210)
    valid &= 0x01010101u;
}
// byte-wise 2-bit fields (first base in the low byte) -> 8 bits, first base most significant
__device__ __forceinline__ uint32_t squeeze4(uint32_t c) {
    return ((c & 0x3u) << 6) | ((c >> 4) & 0x30u) | ((c >> 14) & 0xCu) | (c >> 24);
}

// ConvertBinaySeq (align.cpp:90-162) for one chain: packed words + valid-base mask (01 per ACGT base).
// rw / m5 point at this lane's column of the warp's shared scratch: word j lives at [j * 32].
__device__ __forceinline__ void pack_chain(const uint8_t *sq, uint32_t stride, int len, int chain, uint32_t *rw, uint32_t *m5) {
    if (!chain) {
        const uint2 *q2 = reinterpret_cast<const uint2 *>(sq);          // rows are 8-byte aligned (stride % 8 == 0)
        #pragma unroll 1
        for (int j = 0; j < BSX_FIXWORDS; j++) {
            uint32_t w = 0, m = 0;
            const int nb = len - 16 * j;                                 // bases of the read in this word
            if (nb > 0 && (uint32_t)(16 * j) < stride) {
                const uint2 lo = __ldg(q2 + 2 * j);
                const uint2 hi = (uint32_t)(16 * j + 8) < stride ? __ldg(q2 + 2 * j + 1) : make_uint2(0u, 0u);
                const uint4 q = make_uint4(lo.x, lo.y, hi.x, hi.y);
                uint32_t c, v;
                codes4(q.x, c, v); w = squeeze4(c) << 24; m = squeeze4(v) << 24;
                codes4(q.y, c, v); w |= squeeze4(c) << 16; m |= squeeze4(v) << 16;
                codes4(q.z, c, v); w |= squeeze4(c) << 8; m |= squeeze4(v) << 8;
                codes4(q.w, c, v); w |= squeeze4(c); m |= squeeze4(v);
                if (nb < 16) { const uint32_t keep = ~(0xffffffffu >> (2 * nb)); w &= keep; m &= keep; }   // beyond the read: code 0, invalid
            }
            rw[j * 32] = w; m5[j * 32] = m;
        }
    } else {
        // reversed read through rev_alphabet (param.cpp:215-218): complement; every non-ACGT byte -> 3
        #pragma unroll 1
        for (int j = 0; j < BSX_FIXWORDS; j++) {
            uint32_t w = 0, m = 0;
            #pragma unroll 1
            for (int b = 0; b < 16; b++) {
                const int i = 16 * j + b;
                uint32_t code = 0, v = 0;
                if (i < len) {
                    const uint32_t ch = sq[len - 1 - i], lc = ch | 0x20u;
                    v = (lc == 'a') | (lc == 'c') | (lc == 'g') | (lc == 't');
                    uint32_t x = (ch >> 1) & 3u; x ^= x >> 1;
                    code = v ? 3u - x : 3u;
                }
                w = (w << 2) | code; m = (m << 2) | v;
            }
            rw[j * 32] = w; m5[j * 32] = m;
        }
    }
}

// TrimAdapter (align.cpp:371-425): adapters in -A order, positions ascending, first success wins
__device__ int trim_adapter(const MapArgs &A, const uint8_t *sq, int len) {
    const int s = A.s, tail = MapKernel::rrbs ? 5 : 4;
    #pragma unroll 1
    for (int a = 0; a < A.n_adapter; a++) {
        const int al = A.adapter_len[a];
        #pragma unroll 1
        for (int pos = s; pos < len - tail; pos++) {
            int m0 = 0, k = 0;
            #pragma unroll 1
            for (; k < al && k < 15 && pos + k < len; k++) {
                m0 += (A.adapter[a][k] != (char)sq[pos + k]);
                if (m0 > 4) break;
            }
            bool ok = false;
            if constexpr (!MapKernel::rrbs) ok = (k >= m0 * 5 && k > 3);
            else if (k >= m0 * 5) {
                // digestion-site remnant just before the adapter (align.cpp:383-404)
                const int sl = A.site_len, dp = A.digest_pos;
                int m = m0, m2 = m0;
                #pragma unroll 1
                for (int t = 0; t < sl - dp; t++) {
                    const char x = A.digest_site[t], y = (char)sq[pos - sl + dp + t];
                    m += (x != y) && (x != 'C' || y != 'T');
                    m2 += (x != y) && (x != 'G' || y != 'A');
                }
                ok = (k >= m * 5) || (A.pairend && k >= m2 * 5);
            }
            if (ok) return pos;
        }
    }
    return len;
}

// ---- packed read slots (include/bsmap_b200.h): 2-bit bases, four per byte, then a 1-bit valid mask, eight per byte
// base i of a packed slot: 2-bit code | valid << 2
__device__ __forceinline__ uint32_t pk_base(const uint8_t *pk, uint32_t mask_off, int i) {
    const uint32_t c = (pk[i >> 2] >> (6 - 2 * (i & 3))) & 3u, v = (pk[mask_off + (i >> 3)] >> (7 - (i & 7))) & 1u;
    return c | (v << 2);
}
// 16 mask bits (first base in bit 15) -> 01 per valid base, first base in bits 31:30
__device__ __forceinline__ uint32_t spread16(uint32_t x) {
    x = (x | (x << 8)) & 0x00FF00FFu; x = (x | (x << 4)) & 0x0F0F0F0Fu;
    x = (x | (x << 2)) & 0x33333333u; return (x | (x << 1)) & 0x55555555u;
}

// ConvertBinaySeq from a packed slot: chain 0 is a byte swap and a bit spread, chain 1 walks the read backwards
__device__ __forceinline__ void pack_chain_packed(const uint8_t *pk, uint32_t mask_off, int len, int chain, uint32_t *rw, uint32_t *m5) {
    if (!chain) {
        const uint32_t *w4 = reinterpret_cast<const uint32_t *>(pk);       // slots are 4-byte aligned
        #pragma unroll 1
        for (int j = 0; j < BSX_FIXWORDS; j++) {
            uint32_t w = 0, m = 0;
            const int nb = len - 16 * j;
            if (nb > 0) {
                w = __byte_perm(__ldg(w4 + j), 0u, 0x0123);                 // first base of the word into bits 31:30
                m = spread16(((uint32_t)__ldg(pk + mask_off + 2 * j) << 8) | (uint32_t)__ldg(pk + mask_off + 2 * j + 1));
                if (nb < 16) { const uint32_t keep = ~(0xffffffffu >> (2 * nb)); w &= keep; m &= keep; }
                w &= m | (m << 1);                                          // invalid bases carry code 0 (alphabet[], param.cpp:210)
            }
            rw[j * 32] = w; m5[j * 32] = m;
        }
    } else {
        #pragma unroll 1
        for (int j = 0; j < BSX_FIXWORDS; j++) {
            uint32_t w = 0, m = 0;
            #pragma unroll 1
            for (int b = 0; b < 16; b++) {
                const int i = 16 * j + b;
                uint32_t code = 0, v = 0;
                if (i < len) {
                    const uint32_t x = pk_base(pk, mask_off, len - 1 - i);
                    v = x >> 2;
                    code = v ? 3u - (x & 3u) : 3u;                          // rev_alphabet (param.cpp:215-218)
                }
                w = (w << 2) | code; m = (m << 2) | v;
            }
            rw[j * 32] = w; m5[j * 32] = m;
        }
    }
}

// TrimAdapter on a packed slot.  Adapters and the digestion site are upper-case ACGT (checked on the host), so
// "characters differ" is "invalid base or different code".
__device__ int trim_adapter_packed(const MapArgs &A, const uint8_t *pk, int len) {
    const int s = A.s, tail = MapKernel::rrbs ? 5 : 4;
    const uint32_t mo = A.pk_mask_off;
    #pragma unroll 1
    for (int a = 0; a < A.n_adapter; a++) {
        const int al = A.adapter_len[a];
        #pragma unroll 1
        for (int pos = s; pos < len - tail; pos++) {
            int m0 = 0, k = 0;
            #pragma unroll 1
            for (; k < al && k < 15 && pos + k < len; k++) {
                m0 += (pk_base(pk, mo, pos + k) != (bsx_code_fwd((uint8_t)A.adapter[a][k]) | 4u));
                if (m0 > 4) break;
            }
            bool ok = false;
            if constexpr (!MapKernel::rrbs) ok = (k >= m0 * 5 && k > 3);
            else if (k >= m0 * 5) {
                const int sl = A.site_len, dp = A.digest_pos;
                int m = m0, m2 = m0;
                #pragma unroll 1
                for (int t = 0; t < sl - dp; t++) {
                    const uint32_t x = bsx_code_fwd((uint8_t)A.digest_site[t]) | 4u, y = pk_base(pk, mo, pos - sl + dp + t);
                    m += (x != y) && (x != 5u || y != 7u);                  // 'C' vs 'T'
                    m2 += (x != y) && (x != 6u || y != 4u);                 // 'G' vs 'A'
                }
                ok = (k >= m * 5) || (A.pairend && k >= m2 * 5);
            }
            if (ok) return pos;
        }
    }
    return len;
}

// seed_array[p] (align.cpp:101-105): 3-letter key of the seed starting at read offset p
__device__ __forceinline__ uint32_t seed_key(const MapArgs &A, const uint32_t *rw, int p) {
    const int j = p >> 4, sh = (p & 15) * 2;
    const uint32_t hi = rw[j * 32], lo = (j + 1 < BSX_FIXWORDS) ? rw[(j + 1) * 32] : 0u;
    const uint32_t v = __funnelshift_l(lo, hi, sh) >> (32 - 2 * A.s);
    return bsx_xt(v & A.seed_bits, A.s);
}

// list header of seed key `key`: {list start, reverse-strand start, list end} (tab is the CSR of the seed table)
// A probe is a random 12-byte read of a 344 MB table: fetch 64 bytes from HBM for it, not the default 128-byte line
// (measured in round 1: 121 B of HBM traffic per random gather with the default load, 62 B with .L2::64B).
__device__ __forceinline__ uint3 probe_tab(const MapArgs &A, uint32_t key) {
    uint3 r;
    const uint32_t *p = A.tab + 2 * (size_t)key;
    asm volatile("ld.global.nc.L2::64B.v2.u32 {%0,%1}, [%2];" : "=r"(r.x), "=r"(r.y) : "l"(p));
    asm volatile("ld.global.nc.L2::64B.u32 %0, [%1];" : "=r"(r.z) : "l"(p + 2));
    return r;
}

// RRBS: the table is a CSR over (key, group) (bsx_index.cu); the whole list of a key -- ref.index[key].n1, what
// ReorderSeed ranks the segments by (align.cpp:474-485) -- spans its `groups` consecutive slots
__device__ __forceinline__ uint32_t probe_rrbs_size(const MapArgs &A, uint32_t key) {
    const uint32_t *p = A.tab + (size_t)key * A.rrbs_groups;
    return __ldg(p + A.rrbs_groups) - __ldg(p);
}

// Seed probing and selection for one chain; writes plan[] of the image, returns the number of probes.
// Only the list SIZES are kept per probed offset (a thread-local array goes through L1/L2 to HBM for 5 920 resident
// warps); the bounds of the lists that end up in the plan are read again -- the lines were fetched moments ago.
__device__ __forceinline__ int select_seeds(const MapArgs &A, const PrepSm *K, const uint32_t *rw, int len, int seg, int chain,
                            uint4 *plan, uint32_t *dbg) {
    const int s = A.s, I = A.I;
    constexpr bool rrbs = MapKernel::rrbs;
    const int mo = (rrbs || len - I + 1 < 0) ? 0 : (int)K->remof[len - I + 1];   // max_offset = (len-I+1) % s
    const int cso = (rrbs && chain) ? (int)K->remof[len] : 0;                     // cseed_offset (RRBS rc chain)
    const int lim = I - 1 + mo;
    const int w = min(lim + 1, s);                                                // probed offsets per segment (the last one takes the tail)
    // per probed offset, indexed n*w + (p - n*s): list "size" (index2[key][0])
    uint32_t sz[BSX_MAX_KEYS + 16];
    uint32_t T[16 * 16];
    int arr[16], order[16];
    int np = 0;
    // 1. every read offset that can carry a seed: segment n owns [n*s, n*s + I-1 + max_offset] (profile.a - i lies
    //    in [n*s, n*s+I-1]).  The union of those ranges is probed once, four probes in flight per lane.
    {
        const int total = rrbs ? seg : (seg > 0 ? (seg - 1) * w + lim + 1 : 0);
        int n = 0, r = 0;                                                 // (segment, offset) of flat probe q
        #pragma unroll 1
        for (int q0 = 0; q0 < total; q0 += 4) {
            uint32_t key[4]; uint3 h[4]; bool ok[4];
#pragma unroll
            for (int u = 0; u < 4; u++) {
                const int pofs = rrbs ? cso + n * s : n * s + r;
                ok[u] = (q0 + u < total) && (pofs + s <= len);
                key[u] = ok[u] ? seed_key(A, rw, pofs) : 0u;
                if (rrbs || (r + 1 >= w && n < seg - 1)) { n++; r = 0; } else r++;
            }
#pragma unroll
            for (int u = 0; u < 4; u++) h[u] = !ok[u] ? make_uint3(0u, 0u, 0u) : (rrbs ? make_uint3(0u, 0u, probe_rrbs_size(A, key[u])) : probe_tab(A, key[u]));
#pragma unroll
            for (int u = 0; u < 4; u++) {
                if (q0 + u < total) {
                    const uint32_t cnt = h[u].z - h[u].x;
                    sz[q0 + u] = rrbs ? cnt : (cnt ? cnt + 2 : 0u);      // index2[key][0] = n + 2 (App. B Q7); RRBS: n1
                    np += ok[u];
                }
            }
        }
    }
    // 2. T[n][o] = CountSeeds(n, o) (align.cpp:549-556) for every segment and start offset o <= max_offset
    if (!rrbs) {
        #pragma unroll 1
        for (int n = 0; n < seg; n++)
            #pragma unroll 1
            for (int o = 0; o <= mo; o++) {
                uint32_t tt = 0;
                #pragma unroll 1
                for (int k = 0; k < I; k++) tt += sz[n * w + ((int)K->profA[n * 16 + k] + o - k - n * s)];
                T[n * 16 + o] = tt;
            }
    }
    // 3. ReorderSeed (align.cpp:454-468): global offset = FIRST minimum of GetTotalSeedLoc over [0, max_offset)
    int og = 0;                                  // App. B Q4: defined as 0 when the loop is empty
    if (!rrbs && mo > 1) {
        uint32_t best = 0xffffffffu;
        #pragma unroll 1
        for (int o = 0; o < mo; o++) {
            uint32_t tt = 0;
            #pragma unroll 1
            for (int n = 0; n < seg; n++) tt += T[n * 16 + o];
            if (tt < best) { best = tt; og = o; }
        }
    }
    // AdjustSeedStartArray (align.cpp:506-528)
    #pragma unroll 1
    for (int n = 0; n < seg; n++) arr[n] = og;
    if (!rrbs) {
        #pragma unroll 1
        for (int i = 0; i < seg; i++) {
            const int ptr = (i & 1) == 0 ? i / 2 : seg - 1 - i / 2;
            uint32_t total = 0xffffffffu;
            const int start = (ptr == 0) ? 0 : arr[ptr - 1];
            const int end = (ptr == seg - 1) ? mo : arr[ptr + 1];
            int bi = start;
            #pragma unroll 1
            for (int ii = start; ii <= end; ii++) {
                const uint32_t tt = T[ptr * 16 + ii];
                if (tt < total) { total = tt; bi = ii; }
            }
            arr[ptr] = bi;
        }
    }
    // seedindex: (sum of list sizes, segment) ascending (align.cpp:474-485)
    #pragma unroll 1
    for (int n = 0; n < seg; n++) {
        const uint32_t mine = rrbs ? sz[n] : T[n * 16 + arr[n]];
        int rank = 0;
        #pragma unroll 1
        for (int m = 0; m < seg; m++) {
            const uint32_t other = rrbs ? sz[m] : T[m * 16 + arr[m]];
            rank += (other < mine) || (other == mine && m < n);
        }
        order[rank] = n;
    }
    if (dbg) {
        dbg[chain * 20] = (uint32_t)seg;
        for (int n = 0; n < seg && n < 9; n++) { dbg[chain * 20 + 1 + n] = (uint32_t)arr[n]; dbg[chain * 20 + 10 + n] = (uint32_t)order[n]; }
    }
    // plan[mode][k]: list bounds and read offset of sub-seed k of the segment processed in that mode
    const int per = rrbs ? 1 : I;
    #pragma unroll 1
    for (int m = 0; m < seg; m++) {
        const int sg = order[m];
        #pragma unroll 1
        for (int k = 0; k < per; k++) {
            const int p = rrbs ? (sg * s + cso) : ((int)K->profA[sg * 16 + k] + arr[sg] - k);
            uint3 h = make_uint3(0u, 0u, 0u);
            if (p + s <= len) {
                if (!rrbs) h = probe_tab(A, seed_key(A, rw, p));
                else {
                    // the entries SnpAlign does not skip: segment sg of plain entries for the read as is, segment
                    // len/s - 1 - sg of mirrored entries for its reverse complement (align.cpp:187, 222-229)
                    const uint32_t g = chain ? 2u * (uint32_t)((int)K->segof[len] - 1 - sg) + 1u : 2u * (uint32_t)sg;
                    if (g < A.rrbs_groups) {
                        const uint32_t *t = A.tab + (size_t)seed_key(A, rw, p) * A.rrbs_groups + g;
                        h.x = __ldg(t); h.z = __ldg(t + 1); h.y = h.z;
                    }
                }
            }
            plan[m * per + k] = make_uint4(h.x, h.y, h.z, (uint32_t)p | ((uint32_t)sg << 16));
        }
    }
    return np;
}

// Prepare unit `u` (read r, mate) into the image at `img` (layout: bsx_map.cuh); returns the number of table probes.
// noinline on purpose: called once per 32 units, with its own register allocation.
// rw / m5: this lane's column of the warp's PrepCol (shared memory) -- the packed read is indexed by data-dependent
// word numbers, which as a thread-local array cost one 32-byte sector per access (130 sectors per read).
__device__ __noinline__ int bsx_prep_unit(const MapArgs &A, const PrepSm *Kp, uint32_t *rw, uint32_t *m5, uint32_t u, uint8_t *img) {
    const PrepSm &K = *Kp;
    int np = 0;
    {
        const uint32_t r = A.mates == 2 ? u >> 1 : u;
        const int mate = A.mates == 2 ? (int)(u & 1u) : 0;
        const uint8_t *sq = (mate ? A.seq_b : A.seq_a) + (size_t)r * A.stride;
        int len = (mate ? A.len_b : A.len_a)[r];
        if (len > A.max_readlen) len = A.max_readlen;                       // reads.cpp:115-117
        if (len > BSX_MAX_READLEN) len = BSX_MAX_READLEN;
        if (len > (int)(A.packed ? A.pk_maxlen : A.stride)) len = (int)(A.packed ? A.pk_maxlen : A.stride);
        const int readset = A.mates == 2 ? mate + 1 : A.readset;
        const int raw = len;
        len = A.packed ? trim_adapter_packed(A, sq, len) : trim_adapter(A, sq, len);
        const int fc = A.chains || (readset < 2), cc = A.chains || (readset == 2);   // flag_chain / cflag_chain (align.cpp:93-94)
        int filtered = len < A.s, rmsn = 0, seg = 0;
        if (!filtered) {
            // CountNs (align.cpp:48-55) from the valid-base mask of the chain the read uses first
            if (A.packed) pack_chain_packed(sq, A.pk_mask_off, len, fc ? 0 : 1, rw, m5); else pack_chain(sq, A.stride, len, fc ? 0 : 1, rw, m5);
            int nv = 0;
            #pragma unroll 1
            for (int j = 0; j < BSX_FIXWORDS; j++) nv += __popc(m5[j * 32]);
            if (len - nv > A.max_ns) filtered = 1;
        }
        if (!filtered) {
            // read_max_snp_num = (v+1)*(len-1)/raw_readlen (align.cpp:586); equals v for an untrimmed read longer than v
            rmsn = (len == raw && A.v + 1 <= len) ? A.v : (int)((unsigned)(A.v + 1) * (unsigned)(len - 1) / (unsigned)raw);
            const int q = len - A.I + 1;
            seg = q > 0 ? min((int)K.segof[q], rmsn + 1) : 0;               // seedseg_num (align.cpp:440)
            uint32_t *dbg = A.debug ? A.debug + (size_t)r * 40 : nullptr;
            #pragma unroll 1
            for (int chain = 0; chain < 2; chain++) {
                if (chain == 0 ? !fc : !cc) continue;
                if (chain == 1 && fc) {                                          // -n 1: the other orientation, same scratch
                    if (A.packed) pack_chain_packed(sq, A.pk_mask_off, len, 1, rw, m5); else pack_chain(sq, A.stride, len, 1, rw, m5);
                }
                uint32_t *slot = reinterpret_cast<uint32_t *>(img + sizeof(ImgHdr) + (A.nslot == 2 ? chain : 0) * A.img_slot);
                np += select_seeds(A, &K, rw, len, seg, chain, reinterpret_cast<uint4 *>(slot + 2 * BSX_FIXWORDS), dbg);
                #pragma unroll 1
                for (int j = 0; j < BSX_FIXWORDS; j++) { slot[j] = rw[j * 32]; slot[BSX_FIXWORDS + j] = m5[j * 32]; }
            }
        }
        ImgHdr h;
        h.index = A.first_index + r;
        h.geom = (uint32_t)len | ((uint32_t)rmsn << 8) | ((uint32_t)seg << 16) | ((uint32_t)(filtered | (fc << 1) | (cc << 2)) << 24);
        h.aux = (uint32_t)raw | ((uint32_t)readset << 8);
        h.pad = 0;
        *reinterpret_cast<uint4 *>(img) = *reinterpret_cast<const uint4 *>(&h);
    }
    return np;
}

}  // namespace
