// bsx_api.cu -- the C ABI (include/bsmap_b200.h): handles, batch plumbing, stream pipeline.
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <utility>
#include <vector>
#include "bsx_common.cuh"
#include "bsx_internal.h"
#include "bsx_map.cuh"

// ------------------------------------------------------------------------------------ errors
static thread_local char g_err[1024] = "";
void bsx_set_error(const char *fmt, ...) {
    va_list ap; va_start(ap, fmt); vsnprintf(g_err, sizeof g_err, fmt, ap); va_end(ap);
}
extern "C" const char *bsx_last_error(void) { return g_err; }

extern "C" int bsx_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

static int require_device(int device) {
    int n = bsx_device_count();
    if (n <= 0) { bsx_set_error("no CUDA device available: bsmap_b200 has no CPU fallback"); return BSX_ERR_CUDA; }
    if (device < 0 || device >= n) { bsx_set_error("device %d out of range (have %d)", device, n); return BSX_ERR_ARG; }
    return BSX_OK;
}

// Param::Param (param.cpp:6-83)
extern "C" void bsx_params_default(bsx_params *p) {
    memset(p, 0, sizeof *p);
    p->seed_size = 16; p->index_interval = 4; p->max_snp_num = 2; p->max_num_hits = BSX_MAXHITS;
    p->report_repeat_hits = 1; p->min_insert = 28; p->max_insert = 500; p->max_ns = 5;
    p->max_readlen = BSX_MAX_READLEN;
}

static int check_params(const bsx_params *p) {
    if (p->seed_size < 8 || p->seed_size > 16) { bsx_set_error("seed size must be 8..16 (got %d)", p->seed_size); return BSX_ERR_ARG; }
    if (p->index_interval < 1 || p->index_interval > 16) { bsx_set_error("index interval must be 1..16"); return BSX_ERR_ARG; }
    if (p->max_snp_num < 0 || p->max_snp_num > BSX_MAXSNPS) { bsx_set_error("max mismatches must be 0..%d", BSX_MAXSNPS); return BSX_ERR_ARG; }
    if (p->max_num_hits < 1 || p->max_num_hits > BSX_MAXHITS) { bsx_set_error("max multi-hits must be 1..%d", BSX_MAXHITS); return BSX_ERR_ARG; }
    if (p->n_adapter < 0 || p->n_adapter > BSX_MAX_ADAPTERS) { bsx_set_error("at most %d adapters", BSX_MAX_ADAPTERS); return BSX_ERR_ARG; }
    if (p->rrbs && (p->seed_size != 12 || p->index_interval != 1)) { bsx_set_error("RRBS mode forces seed 12 / interval 1 (param.cpp:95-106)"); return BSX_ERR_ARG; }
    return BSX_OK;
}

// ------------------------------------------------------------------------------------ index
extern "C" int bsx_index_create(const bsx_params *p, int n_seq, const char *const *names,
                                const char *const *seqs, const uint32_t *lens, int device, bsx_index **out) {
    if (!p || !out || n_seq <= 0 || !names || !seqs || !lens) { bsx_set_error("bsx_index_create: bad argument"); return BSX_ERR_ARG; }
    int rc = check_params(p); if (rc) return rc;
    rc = require_device(device); if (rc) return rc;
    bsx_index *ix = new bsx_index();
    ix->device = device; ix->par = *p; ix->n_seq = (uint32_t)n_seq;
    for (int k = 0; k < n_seq; k++) { ix->names.emplace_back(names[k]); ix->size.push_back(lens[k]); }
    rc = bsx_index_build_device(ix, seqs);
    if (rc) { bsx_index_free_device(ix); delete ix; return rc; }
    *out = ix;
    return BSX_OK;
}

// ---- packed reference cache (SURVEY §8 f2).  The seed table takes 0.4 s of kernels to rebuild, so what is worth
// keeping on disk is what the rebuild needs and the FASTA makes expensive: the packed forward strand (a quarter of
// the text), the UnmaskRegion blocks, names and sizes.  Parameter-independent (WGBS); the rc strand and the table
// are derived on the device at load.
namespace {
struct PackedHeader { char magic[8]; uint32_t version, n_seq; uint64_t n_words, n_blocks, names_bytes; };
}

extern "C" int bsx_index_save_packed(const bsx_index *ix, const char *path) {
    if (!ix || !path || ix->device < 0) { bsx_set_error("bsx_index_save_packed: bad argument"); return BSX_ERR_ARG; }
    if (ix->par.rrbs) { bsx_set_error("bsx_index_save_packed: RRBS indexes are not cached (digestion sites need the text)"); return BSX_ERR_ARG; }
    BSX_CUDA_CHECK(cudaSetDevice(ix->device));
    std::vector<uint32_t> ref(ix->n_words);
    BSX_CUDA_CHECK(cudaMemcpy(ref.data(), ix->d_refcat, ix->n_words * 4, cudaMemcpyDeviceToHost));
    std::string names;
    for (const std::string &n : ix->names) { names += n; names.push_back('\0'); }
    PackedHeader h; memset(&h, 0, sizeof h);
    memcpy(h.magic, "BSXPACK", 8); h.version = 1; h.n_seq = ix->n_seq; h.n_words = ix->n_words; h.n_blocks = ix->blocks.size(); h.names_bytes = names.size();
    const std::string tmp = std::string(path) + ".tmp";
    FILE *f = fopen(tmp.c_str(), "wb");
    if (!f) { bsx_set_error("bsx_index_save_packed: cannot write %s", tmp.c_str()); return BSX_ERR_IO; }
    bool ok = fwrite(&h, sizeof h, 1, f) == 1 && fwrite(names.data(), 1, names.size(), f) == names.size() &&
              fwrite(ix->size.data(), 4, ix->n_seq, f) == ix->n_seq &&
              (ix->blocks.empty() || fwrite(ix->blocks.data(), sizeof(bsx_block), ix->blocks.size(), f) == ix->blocks.size()) &&
              fwrite(ref.data(), 4, ref.size(), f) == ref.size();
    ok = (fclose(f) == 0) && ok;
    if (!ok || rename(tmp.c_str(), path) != 0) { remove(tmp.c_str()); bsx_set_error("bsx_index_save_packed: write to %s failed", path); return BSX_ERR_IO; }
    return BSX_OK;
}

extern "C" int bsx_index_create_from_packed(const bsx_params *p, const char *path, int device, bsx_index **out) {
    if (!p || !path || !out) { bsx_set_error("bsx_index_create_from_packed: bad argument"); return BSX_ERR_ARG; }
    int rc = check_params(p); if (rc) return rc;
    if (p->rrbs) { bsx_set_error("a packed reference cache cannot seed an RRBS index (digestion sites need the text)"); return BSX_ERR_ARG; }
    rc = require_device(device); if (rc) return rc;
    FILE *f = fopen(path, "rb");
    if (!f) { bsx_set_error("cannot open packed reference %s", path); return BSX_ERR_IO; }
    PackedHeader h;
    bsx_index *ix = new bsx_index();
    auto fail = [&](const char *why) { fclose(f); bsx_index_free_device(ix); delete ix; bsx_set_error("%s: %s", path, why); return BSX_ERR_IO; };
    if (fread(&h, sizeof h, 1, f) != 1 || memcmp(h.magic, "BSXPACK", 8) != 0 || h.version != 1) return fail("not a packed reference (BSXPACK v1)");
    std::string names(h.names_bytes, '\0');
    ix->device = device; ix->par = *p; ix->n_seq = h.n_seq;
    ix->size.resize(h.n_seq); ix->blocks.resize(h.n_blocks);
    uint32_t *ref = nullptr;
    if (cudaHostAlloc(&ref, h.n_words * 4, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); return fail("out of pinned host memory"); }
    const bool ok = fread(&names[0], 1, names.size(), f) == names.size() && fread(ix->size.data(), 4, h.n_seq, f) == h.n_seq &&
                    (h.n_blocks == 0 || fread(ix->blocks.data(), sizeof(bsx_block), h.n_blocks, f) == h.n_blocks) &&
                    fread(ref, 4, h.n_words, f) == h.n_words;
    if (!ok) { cudaFreeHost(ref); return fail("truncated file"); }
    for (size_t q = 0; q < names.size() && ix->names.size() < h.n_seq;) { ix->names.emplace_back(names.c_str() + q); q += ix->names.back().size() + 1; }
    if (ix->names.size() != h.n_seq) { cudaFreeHost(ref); return fail("corrupt name table"); }
    fclose(f);
    rc = bsx_index_build_device(ix, nullptr, ref);
    if (rc == BSX_OK && ix->n_words != h.n_words) { bsx_set_error("%s: geometry mismatch", path); rc = BSX_ERR_IO; }
    cudaFreeHost(ref);
    if (rc) { bsx_index_free_device(ix); delete ix; return rc; }
    *out = ix;
    return BSX_OK;
}

// Packed reference only (both strands, anchors, sizes) on the device: what bsx_meth needs; no seed table, cannot map.
extern "C" int bsx_index_create_packed(int n_seq, const char *const *names, const char *const *seqs, const uint32_t *lens,
                                       int device, bsx_index **out) {
    if (!out || n_seq <= 0 || !names || !seqs || !lens) { bsx_set_error("bsx_index_create_packed: bad argument"); return BSX_ERR_ARG; }
    int rc = require_device(device); if (rc) return rc;
    bsx_index *ix = new bsx_index();
    bsx_params_default(&ix->par);
    ix->device = device; ix->n_seq = (uint32_t)n_seq; ix->ref_only = true;
    for (int k = 0; k < n_seq; k++) { ix->names.emplace_back(names[k]); ix->size.push_back(lens[k]); }
    rc = bsx_index_build_device(ix, seqs);
    if (rc) { bsx_index_free_device(ix); delete ix; return rc; }
    *out = ix;
    return BSX_OK;
}

// Host-only index for the text layer: names, sizes, anchors, the packed Watson strand (XR:Z / BSP
// refseq column) and RRBS digestion sites.  It cannot map (device = -1); it exists so that records
// produced on a GPU node can be formatted elsewhere, and so the formatter is testable without a GPU.
extern "C" int bsx_index_create_text_only(const bsx_params *p, int n_seq, const char *const *names,
                                          const char *const *seqs, const uint32_t *lens, bsx_index **out) {
    if (!p || !out || n_seq <= 0 || !names || !seqs || !lens) { bsx_set_error("bsx_index_create_text_only: bad argument"); return BSX_ERR_ARG; }
    bsx_index *ix = new bsx_index();
    ix->device = -1; ix->par = *p; ix->n_seq = (uint32_t)n_seq;
    uint64_t tot = 0;
    ix->anchor.resize(n_seq + 1);
    for (int k = 0; k < n_seq; k++) {
        ix->names.emplace_back(names[k]); ix->size.push_back(lens[k]);
        ix->nwords.push_back((lens[k] + BSX_SEGLEN - 1) / BSX_SEGLEN + 2);
        ix->rc_offset.push_back(ix->nwords[k] * BSX_SEGLEN);
        ix->anchor[k] = (uint32_t)((tot + BSX_REF_MARGIN) * BSX_SEGLEN);
        tot += ix->nwords[k];
    }
    ix->anchor[n_seq] = (uint32_t)((tot + BSX_REF_MARGIN) * BSX_SEGLEN);
    ix->n_words = tot + 2 * BSX_REF_MARGIN;
    ix->h_refcat.assign(ix->n_words, 0);
    ix->sites.assign(n_seq, {});
    const int sl = (int)strnlen(p->digest_site, sizeof p->digest_site);
    for (int k = 0; k < n_seq; k++) {
        uint32_t *w = ix->h_refcat.data() + (ix->anchor[k] >> 4);
        const uint8_t *sq = (const uint8_t *)seqs[k];
        for (uint32_t i = 0; i < lens[k]; i++) w[i >> 4] |= bsx_code_fwd(sq[i]) << (30 - 2 * (i & 15));
        if (p->rrbs)
            for (uint32_t q = 0; q + sl <= lens[k]; q++) {
                bool ok = true;
                for (int t = 0; t < sl; t++) { uint8_t c = sq[q + t]; if (c >= 'a' && c <= 'z') c -= 32; if (c != (uint8_t)p->digest_site[t]) { ok = false; break; } }
                if (ok) ix->sites[k].push_back(q + p->digest_pos);
            }
    }
    *out = ix;
    return BSX_OK;
}

// RefSeq::LoadNextSeq (dbseq.cpp:18-54): name = first token after '>', sequence = whitespace-free
// concatenation of the following tokens up to the next '>' (bsx_load_fasta, bsx_reads.cpp)
extern "C" int bsx_index_create_from_fasta(const bsx_params *p, const char *path, int device, bsx_index **out) {
    std::vector<std::string> names, seqs;
    const int rc = bsx_load_fasta(path, names, seqs);
    if (rc != BSX_OK) return rc;
    std::vector<const char *> np, sp; std::vector<uint32_t> ln;
    for (size_t k = 0; k < seqs.size(); k++) { np.push_back(names[k].c_str()); sp.push_back(seqs[k].data()); ln.push_back((uint32_t)seqs[k].size()); }
    return bsx_index_create(p, (int)seqs.size(), np.data(), sp.data(), ln.data(), device, out);
}

extern "C" int bsx_index_create_text_only_from_fasta(const bsx_params *p, const char *path, bsx_index **out) {
    std::vector<std::string> names, seqs;
    const int rc = bsx_load_fasta(path, names, seqs);
    if (rc != BSX_OK) return rc;
    std::vector<const char *> np, sp; std::vector<uint32_t> ln;
    for (size_t k = 0; k < seqs.size(); k++) { np.push_back(names[k].c_str()); sp.push_back(seqs[k].data()); ln.push_back((uint32_t)seqs[k].size()); }
    return bsx_index_create_text_only(p, (int)seqs.size(), np.data(), sp.data(), ln.data(), out);
}

extern "C" int bsx_index_destroy(bsx_index *ix) {
    if (!ix) return BSX_OK;
    bsx_index_free_device(ix);
    delete ix;
    return BSX_OK;
}

extern "C" int bsx_index_get_info(const bsx_index *ix, bsx_index_info *info) {
    if (!ix || !info) return BSX_ERR_ARG;
    info->n_words = ix->n_words; info->n_keys = ix->n_keys; info->n_entries = ix->n_entries;
    info->n_seq = ix->n_seq; info->device = ix->device; info->build_seconds = ix->build_seconds;
    info->n_tab = ix->ref_only ? 0 : bsx_tab_len(ix);
    info->ctx_words = ix->ref_only ? 0u : (uint32_t)(bsx_ctx_entry_bytes(ix) / 4);
    return BSX_OK;
}
extern "C" const char *bsx_index_seq_name(const bsx_index *ix, uint32_t k) { return (ix && k < ix->n_seq) ? ix->names[k].c_str() : ""; }
extern "C" uint32_t bsx_index_seq_size(const bsx_index *ix, uint32_t k) { return (ix && k < ix->n_seq) ? ix->size[k] : 0; }

extern "C" int bsx_index_download(const bsx_index *ix, int what, void *dst, size_t bytes) {
    if (!ix || !dst) return BSX_ERR_ARG;
    if (ix->device < 0) {   // text-only index: the packed Watson strand is all it has
        if (what != 0 || bytes > ix->h_refcat.size() * 4) { bsx_set_error("text-only index has no device arrays"); return BSX_ERR_ARG; }
        memcpy(dst, ix->h_refcat.data(), bytes);
        return BSX_OK;
    }
    BSX_CUDA_CHECK(cudaSetDevice(ix->device));
    const void *src = nullptr; size_t have = 0;
    switch (what) {
        case 0: src = ix->d_refcat; have = ix->n_words * 4; break;
        case 1: src = ix->d_crefcat; have = ix->n_words * 4; break;
        case 2: src = ix->d_seqinfo; have = ((size_t)ix->n_seq + 1) * 4; break;
        case 3: src = ix->d_tab; have = bsx_tab_len(ix) * 4; break;
        case 4: src = ix->d_pos; have = ix->n_entries * 4; break;
        case 5: src = ix->d_tag; have = ix->d_tag ? ix->n_entries * 4 : 0; break;
        case 6: src = ix->d_ctx; have = ix->d_ctx ? ix->n_entries * bsx_ctx_entry_bytes(ix) : 0; break;
        default: bsx_set_error("bsx_index_download: unknown array %d", what); return BSX_ERR_ARG;
    }
    if (bytes > have) { bsx_set_error("bsx_index_download: asked %zu bytes, array has %zu", bytes, have); return BSX_ERR_ARG; }
    if (bytes) BSX_CUDA_CHECK(cudaMemcpy(dst, src, bytes, cudaMemcpyDeviceToHost));
    return BSX_OK;
}

extern "C" int bsx_index_device_buffers(const bsx_index *ix, void **ptrs, size_t *bytes, int cap) {
    if (!ix || cap < 7) return 0;
    ptrs[0] = ix->d_refcat; bytes[0] = ix->n_words * 4;
    ptrs[1] = ix->d_crefcat; bytes[1] = ix->n_words * 4;
    ptrs[2] = ix->d_tab; bytes[2] = bsx_tab_len(ix) * 4;
    ptrs[3] = ix->d_pos; bytes[3] = ix->n_entries * 4;
    ptrs[4] = ix->d_tag; bytes[4] = ix->d_tag ? ix->n_entries * 4 : 0;
    ptrs[5] = ix->d_ctx; bytes[5] = ix->d_ctx ? ix->n_entries * bsx_ctx_entry_bytes(ix) : 0;
    ptrs[6] = nullptr; bytes[6] = 0;    // (round 1 kept the outer context bases in a second array)
    return 7;
}

// metadata blob: everything a replica needs besides the big device arrays
static void put(std::vector<uint8_t> &b, const void *p, size_t n) { const uint8_t *q = (const uint8_t *)p; b.insert(b.end(), q, q + n); }
static std::vector<uint8_t> meta_blob(const bsx_index *ix) {
    std::vector<uint8_t> b;
    const uint64_t magic = 0x3130585342ULL;  // "BSX01"
    put(b, &magic, 8); put(b, &ix->par, sizeof ix->par);
    put(b, &ix->n_seq, 4); put(b, &ix->n_words, 8); put(b, &ix->n_keys, 8); put(b, &ix->n_entries, 8);
    for (uint32_t k = 0; k < ix->n_seq; k++) {
        uint32_t l = (uint32_t)ix->names[k].size(); put(b, &l, 4); put(b, ix->names[k].data(), l);
        put(b, &ix->size[k], 4); put(b, &ix->rc_offset[k], 4); put(b, &ix->nwords[k], 4); put(b, &ix->anchor[k], 4);
        uint32_t ns = ix->par.rrbs ? (uint32_t)ix->sites[k].size() : 0; put(b, &ns, 4);
        if (ns) put(b, ix->sites[k].data(), (size_t)ns * 4);
    }
    put(b, &ix->anchor[ix->n_seq], 4);
    return b;
}
extern "C" size_t bsx_index_meta_size(const bsx_index *ix) { return ix ? meta_blob(ix).size() : 0; }
extern "C" int bsx_index_meta_export(const bsx_index *ix, void *dst, size_t bytes) {
    if (!ix || !dst) return BSX_ERR_ARG;
    std::vector<uint8_t> b = meta_blob(ix);
    if (bytes < b.size()) { bsx_set_error("meta buffer too small"); return BSX_ERR_ARG; }
    memcpy(dst, b.data(), b.size());
    return BSX_OK;
}
extern "C" int bsx_index_create_shell(const void *meta, size_t bytes, int device, bsx_index **out) {
    if (!meta || !out) return BSX_ERR_ARG;
    int rc = require_device(device); if (rc) return rc;
    const uint8_t *q = (const uint8_t *)meta, *end = q + bytes;
    auto get = [&](void *p, size_t n) { if (q + n > end) return false; memcpy(p, q, n); q += n; return true; };
    uint64_t magic = 0;
    bsx_index *ix = new bsx_index();
    bool ok = get(&magic, 8) && magic == 0x3130585342ULL && get(&ix->par, sizeof ix->par) && get(&ix->n_seq, 4) &&
              get(&ix->n_words, 8) && get(&ix->n_keys, 8) && get(&ix->n_entries, 8);
    if (ok) {
        ix->size.resize(ix->n_seq); ix->rc_offset.resize(ix->n_seq); ix->nwords.resize(ix->n_seq); ix->anchor.resize(ix->n_seq + 1);
        ix->names.resize(ix->n_seq); ix->sites.resize(ix->n_seq);
        for (uint32_t k = 0; ok && k < ix->n_seq; k++) {
            uint32_t l = 0, ns = 0;
            ok = get(&l, 4); if (!ok) break;
            ix->names[k].resize(l); ok = get(&ix->names[k][0], l) && get(&ix->size[k], 4) && get(&ix->rc_offset[k], 4) &&
                                         get(&ix->nwords[k], 4) && get(&ix->anchor[k], 4) && get(&ns, 4);
            if (ok && ns) { ix->sites[k].resize(ns); ok = get(ix->sites[k].data(), (size_t)ns * 4); }
        }
        ok = ok && get(&ix->anchor[ix->n_seq], 4);
    }
    if (!ok) { delete ix; bsx_set_error("bsx_index_create_shell: corrupt metadata"); return BSX_ERR_ARG; }
    ix->device = device;
    rc = bsx_index_alloc_device(ix);
    if (rc) { bsx_index_free_device(ix); delete ix; return rc; }
    *out = ix;
    return BSX_OK;
}

// one-time replica over NVLink (peer copy); the only inter-GPU traffic of the whole design
extern "C" int bsx_index_replicate(const bsx_index *src, int device, bsx_index **out) {
    if (!src || !out) return BSX_ERR_ARG;
    std::vector<uint8_t> b = meta_blob(src);
    int rc = bsx_index_create_shell(b.data(), b.size(), device, out);
    if (rc) return rc;
    void *sp[7], *dp[7]; size_t sb[7], db[7];
    bsx_index_device_buffers(src, sp, sb, 7); bsx_index_device_buffers(*out, dp, db, 7);
    int can = 0;
    cudaDeviceCanAccessPeer(&can, device, src->device);
    if (can) { cudaSetDevice(device); cudaDeviceEnablePeerAccess(src->device, 0); cudaGetLastError(); }
    for (int i = 0; i < 7; i++)
        if (sb[i] && sp[i]) BSX_CUDA_CHECK(cudaMemcpyPeer(dp[i], device, sp[i], src->device, sb[i]));
    BSX_CUDA_CHECK(cudaDeviceSynchronize());
    return BSX_OK;
}

// ------------------------------------------------------------------------------------ mapper
struct bsx_slot {
    cudaStream_t stream = nullptr;
    uint8_t *d_seq_a = nullptr, *d_seq_b = nullptr;
    uint16_t *d_len_a = nullptr, *d_len_b = nullptr;
    bsx_rec *d_out_a = nullptr, *d_out_b = nullptr;
    bsx_pair_rec *d_out_pair = nullptr;
    uint16_t *d_cnt_a = nullptr, *d_cnt_b = nullptr;
    uint32_t *d_counter = nullptr;
    uint2 *d_hits = nullptr; uint32_t *d_dd = nullptr; uint4 *d_pairs = nullptr;
    uint8_t *d_prep = nullptr;   // prepared-read images of one chunk (bsx_prep.cu)
    bool packed = false;         // the slot's read buffers hold packed slots (bsx_packed_stride) instead of ASCII
};

// one of the six mapping kernels with the persistent grid it runs in
struct map_launch {
    const void *kernel = nullptr;
    int n_ctas = 0, warps = BSX_WARPS_PER_CTA;   // warps per CTA: fewer when the plan of a read is large
    size_t smem = 0;                             // dynamic shared memory per CTA
};

struct bsx_mapper {
    const bsx_index *ix = nullptr;
    int device = 0;                  // kept here too: a mapper may be destroyed after its index (garbage-collected bindings)
    bsx_params par{};
    uint32_t max_batch = 0, stride = 0;
    int plan_cap = 0, nslot = 1;
    map_launch se, pe;               // single-end and paired-end kernel of this parameter set and index
    uint32_t hit_stride = 0, dd_stride = 0, pair_stride = 0;
    bool pe_ready = false;
    bsx_slot slot[2];
    unsigned long long *d_stats = nullptr;
    uint32_t *d_debug = nullptr;
    uint64_t launches = 0;
    MapArgs base{};
    bsx_meth *meth = nullptr;        // attached methylation counters: every mapped batch is piled up on its stream
    bsx_meth_opts meth_opts{};
    int meth_sam = 1;
};

// the six mapping kernels (bsx_map_{se,pe}{,_rrbs,_wide}.cu)
extern const void *const bsx_map_se_wgbs, *const bsx_map_se_rrbs, *const bsx_map_se_wide;
extern const void *const bsx_map_pe_wgbs, *const bsx_map_pe_rrbs, *const bsx_map_pe_wide;

static const void *map_kernel(bool pe, bool rrbs, bool wide) {
    if (rrbs) return pe ? bsx_map_pe_rrbs : bsx_map_se_rrbs;
    if (wide) return pe ? bsx_map_pe_wide : bsx_map_se_wide;
    return pe ? bsx_map_pe_wgbs : bsx_map_se_wgbs;
}

// Lets `kernel` launch with `smem` bytes of dynamic shared memory on the current device.  The limit belongs to (kernel,
// device) and is shared by every mapper and host thread, so it is only ever raised: lowering it for one mapper would
// make the launches of another that needs more fail.
static int raise_smem_limit(const void *kernel, size_t smem) {
    static std::mutex mu;
    static std::map<std::pair<const void *, int>, size_t> limit;
    int dev = 0;
    BSX_CUDA_CHECK(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lock(mu);
    size_t &cur = limit[{kernel, dev}];
    if (smem > cur) {
        BSX_CUDA_CHECK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        cur = smem;
    }
    return BSX_OK;
}

// Chooses the kernel for a parameter set and the CTA shape of its persistent grid: eight warps per CTA; a parameter set
// whose per-read plan is large (many segments x -I, -n 1, wide context) runs with fewer.  Fails when none fits on an SM.
static int plan_launch(map_launch &k, bool pe, const bsx_mapper *m, bool wide, int sms) {
    k.kernel = map_kernel(pe, m->par.rrbs, wide);
    for (int w = BSX_WARPS_PER_CTA; w >= 1; w >>= 1) {
        const size_t smem = bsx_cta_smem_bytes(pe ? 2 : 1, m->plan_cap, m->nslot, wide, m->par.rrbs, w);
        if (smem > BSX_MAX_CTA_SMEM) continue;
        int occ = 0;   // resident CTAs per SM
        if (raise_smem_limit(k.kernel, smem) != BSX_OK ||
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k.kernel, w * 32, smem) != cudaSuccess) { cudaGetLastError(); occ = 0; }
        k.warps = w; k.smem = smem; k.n_ctas = sms * occ;
        if (occ >= 1) return BSX_OK;
    }
    bsx_set_error("mapping kernel does not fit on an SM (shared memory: plan of %d entries x %d chains)", m->plan_cap, m->nslot);
    return BSX_ERR_CUDA;
}

static int launch_map(const map_launch &k, const MapArgs &a, cudaStream_t st) {
    int rc = raise_smem_limit(k.kernel, k.smem); if (rc) return rc;
    void *args[] = {const_cast<MapArgs *>(&a)};
    cudaLaunchKernel(k.kernel, dim3(k.n_ctas), dim3(k.warps * 32), args, k.smem, st);
    BSX_CUDA_CHECK(cudaGetLastError());       // the launch's error, cleared so that it does not surface in a later call
    return BSX_OK;
}

static void slot_free(bsx_slot &s) {
    cudaFree(s.d_seq_a); cudaFree(s.d_seq_b); cudaFree(s.d_len_a); cudaFree(s.d_len_b); cudaFree(s.d_out_a); cudaFree(s.d_out_b);
    cudaFree(s.d_out_pair); cudaFree(s.d_cnt_a); cudaFree(s.d_cnt_b); cudaFree(s.d_counter); cudaFree(s.d_hits); cudaFree(s.d_dd); cudaFree(s.d_pairs); cudaFree(s.d_prep);
    if (s.stream) cudaStreamDestroy(s.stream);
    s = bsx_slot();
}

extern "C" int bsx_mapper_destroy(bsx_mapper *m) {
    if (!m) return BSX_OK;
    cudaSetDevice(m->device);
    cudaDeviceSynchronize();
    slot_free(m->slot[0]); slot_free(m->slot[1]);
    cudaFree(m->d_stats); cudaFree(m->d_debug);
    delete m;
    return BSX_OK;
}

static int alloc_pe(bsx_mapper *m) {
    // second mate + pair buckets: allocated on first paired-end use
    if (m->pe_ready) return BSX_OK;
    const size_t warps = (size_t)m->pe.n_ctas * m->pe.warps;
    const uint32_t W1 = (uint32_t)m->par.max_num_hits + 1, lv = (uint32_t)m->par.max_snp_num + 1;
    for (int i = 0; i < 2; i++) {
        bsx_slot &s = m->slot[i];
        BSX_CUDA_CHECK(cudaMalloc(&s.d_seq_b, (size_t)m->max_batch * m->stride));
        BSX_CUDA_CHECK(cudaMalloc(&s.d_len_b, (size_t)m->max_batch * 2));
        BSX_CUDA_CHECK(cudaMalloc(&s.d_out_b, (size_t)m->max_batch * sizeof(bsx_rec)));
        BSX_CUDA_CHECK(cudaMalloc(&s.d_cnt_b, (size_t)m->max_batch * 32));
        BSX_CUDA_CHECK(cudaMalloc(&s.d_out_pair, (size_t)m->max_batch * sizeof(bsx_pair_rec)));
        // all-level hit storage for both mates replaces the SE scratch
        cudaFree(s.d_hits); cudaFree(s.d_dd); s.d_hits = nullptr; s.d_dd = nullptr;
        const size_t se_warps = (size_t)m->se.n_ctas * m->se.warps;
        const size_t hit_elems = std::max(warps * 2 * (size_t)(lv * 2 * W1), se_warps * (size_t)(2 * W1));
        const size_t dd_elems = std::max(warps * 2, se_warps) * (size_t)m->dd_stride;
        BSX_CUDA_CHECK(cudaMalloc(&s.d_hits, hit_elems * sizeof(uint2)));
        BSX_CUDA_CHECK(cudaMalloc(&s.d_dd, dd_elems * 4));
        BSX_CUDA_CHECK(cudaMalloc(&s.d_pairs, warps * (size_t)m->pair_stride * sizeof(uint4)));
    }
    m->pe_ready = true;
    return BSX_OK;
}

static int mapper_init(bsx_mapper *m, const bsx_index *ix, const bsx_params *p, uint32_t max_batch, uint32_t stride);

extern "C" int bsx_mapper_create(const bsx_index *ix, const bsx_params *p, uint32_t max_batch, uint32_t stride, bsx_mapper **out) {
    if (!ix || !p || !out || max_batch == 0) { bsx_set_error("bsx_mapper_create: bad argument"); return BSX_ERR_ARG; }
    if (ix->device < 0) { bsx_set_error("text-only index cannot map: build it with bsx_index_create on a CUDA device"); return BSX_ERR_CUDA; }
    if (ix->ref_only) { bsx_set_error("packed-reference index (bsx_index_create_packed) has no seed table and cannot map"); return BSX_ERR_ARG; }
    int rc = check_params(p); if (rc) return rc;
    if (stride % 8 != 0 || stride < 16) { bsx_set_error("read stride must be a multiple of 8, at least 16 (got %u)", stride); return BSX_ERR_ARG; }
    if (p->seed_size != ix->par.seed_size || p->index_interval != ix->par.index_interval || p->rrbs != ix->par.rrbs) {
        bsx_set_error("mapper parameters (-s/-I/-D) differ from the index they were built with"); return BSX_ERR_ARG; }
    if (p->rrbs && (p->pairend || p->chains) != (ix->par.pairend || ix->par.chains)) {
        bsx_set_error("RRBS index was built for a different strand set (-b/-n)"); return BSX_ERR_ARG; }
    rc = require_device(ix->device); if (rc) return rc;
    BSX_CUDA_CHECK(cudaSetDevice(ix->device));
    bsx_mapper *m = new bsx_mapper();
    m->ix = ix; m->device = ix->device;
    rc = mapper_init(m, ix, p, max_batch, stride);
    if (rc != BSX_OK) { bsx_mapper_destroy(m); return rc; }     // frees whatever was allocated before the failure
    *out = m;
    return BSX_OK;
}

static int mapper_init(bsx_mapper *m, const bsx_index *ix, const bsx_params *p, uint32_t max_batch, uint32_t stride) {
    m->ix = ix; m->device = ix->device; m->par = *p; m->max_batch = max_batch; m->stride = stride;
    int readlen = std::min(p->max_readlen, BSX_MAX_READLEN);
    int maxseg = std::min((readlen - p->index_interval + 1) / p->seed_size, p->max_snp_num + 1);
    if (maxseg < 1) maxseg = 1;
    m->plan_cap = maxseg * (p->rrbs ? 1 : p->index_interval);
    m->nslot = p->chains ? 2 : 1;
    int sms = 0;
    BSX_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ix->device));
    // the kernel follows the index layout: an index built with -v >= 8 holds 16-byte context entries whatever -v the mapper uses
    const bool wide = !p->rrbs && ix->ctx_wide;
    int rc = plan_launch(m->se, false, m, wide, sms); if (rc) return rc;
    rc = plan_launch(m->pe, true, m, wide, sms); if (rc) return rc;
    const uint32_t W1 = (uint32_t)p->max_num_hits + 1, lv = (uint32_t)p->max_snp_num + 1;
    m->hit_stride = 2 * W1;                        // SE: only the best level is kept
    m->dd_stride = lv * (uint32_t)p->max_num_hits + 32;
    m->pair_stride = (2 * (uint32_t)p->max_snp_num + 1) * W1 * 2;   // uint4 units (32-byte PairHit)
    const size_t se_warps = (size_t)m->se.n_ctas * m->se.warps;
    // prepared-unit images: 32 per resident warp (phase A of the align kernels, bsx_prep.cuh)
    const size_t prep_bytes = std::max(se_warps, (size_t)m->pe.n_ctas * m->pe.warps) * 32u * bsx_image_bytes(m->plan_cap, m->nslot);
    for (int i = 0; i < 2; i++) {
        bsx_slot &s = m->slot[i];
        BSX_CUDA_CHECK(cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking));
        BSX_CUDA_CHECK(cudaMalloc(&s.d_seq_a, (size_t)max_batch * stride));
        BSX_CUDA_CHECK(cudaMalloc(&s.d_len_a, (size_t)max_batch * 2));
        BSX_CUDA_CHECK(cudaMalloc(&s.d_out_a, (size_t)max_batch * sizeof(bsx_rec)));
        BSX_CUDA_CHECK(cudaMalloc(&s.d_cnt_a, (size_t)max_batch * 32));
        BSX_CUDA_CHECK(cudaMalloc(&s.d_counter, 64));
        BSX_CUDA_CHECK(cudaMalloc(&s.d_hits, se_warps * (size_t)m->hit_stride * sizeof(uint2)));
        BSX_CUDA_CHECK(cudaMalloc(&s.d_dd, se_warps * (size_t)m->dd_stride * 4));
        BSX_CUDA_CHECK(cudaMalloc(&s.d_prep, prep_bytes));
        BSX_CUDA_CHECK(cudaMemset(s.d_prep, 0, prep_bytes));
    }
    BSX_CUDA_CHECK(cudaMalloc(&m->d_stats, 8 * sizeof(unsigned long long)));
    BSX_CUDA_CHECK(cudaMemset(m->d_stats, 0, 8 * sizeof(unsigned long long)));
    if (getenv("BSX_DEBUG_SEEDS")) {
        BSX_CUDA_CHECK(cudaMalloc(&m->d_debug, (size_t)max_batch * 40 * 4));
        BSX_CUDA_CHECK(cudaMemset(m->d_debug, 0, (size_t)max_batch * 40 * 4));
    }
    MapArgs &a = m->base;
    memset(&a, 0, sizeof a);
    a.refcat = ix->d_refcat; a.crefcat = ix->d_crefcat; a.tab = ix->d_tab; a.pos = ix->d_pos; a.tag = ix->d_tag; a.ctx = ix->d_ctx;
    a.ctx_wide = ix->ctx_wide ? 1 : 0;
    a.seqinfo = ix->d_seqinfo; a.sites = ix->d_sites; a.site_off = ix->d_site_off; a.n_seq = ix->n_seq;
    a.s = p->seed_size; a.I = p->index_interval; a.v = p->max_snp_num; a.W = p->max_num_hits; a.r = p->report_repeat_hits;
    a.min_insert = p->min_insert; a.max_insert = p->max_insert; a.chains = p->chains; a.pairend = p->pairend; a.rrbs = p->rrbs;
    a.randseed = p->randseed; a.max_ns = p->max_ns; a.max_readlen = p->max_readlen; a.n_adapter = p->n_adapter;
    a.site_len = (int)strnlen(p->digest_site, sizeof p->digest_site); a.digest_pos = p->digest_pos;
    a.seed_bits = (p->seed_size == 16) ? 0xffffffffu : ((1u << (2 * p->seed_size)) - 1);
    a.rrbs_groups = bsx_rrbs_groups(p->seed_size);
    a.plan_cap = m->plan_cap; a.nslot = m->nslot;
    bsx_map_args_derive(a);
    for (int i = 0; i < p->n_adapter; i++) { a.adapter_len[i] = (int)strnlen(p->adapter[i], 63); memcpy(a.adapter[i], p->adapter[i], 64); }
    memcpy(a.digest_site, p->digest_site, sizeof a.digest_site);
    a.stride = stride; a.stats = m->d_stats; a.debug = m->d_debug;
    a.hit_stride = m->hit_stride; a.dd_stride = m->dd_stride; a.pair_stride = m->pair_stride;
    return BSX_OK;
}

static cudaStream_t pick_stream(bsx_mapper *m, int slot, void *stream) { return stream ? (cudaStream_t)stream : m->slot[slot].stream; }

// packed input needs what the device compares against to be upper-case ACGT (include/bsmap_b200.h)
static int check_packed_ok(const bsx_mapper *m) {
    auto acgt = [](const char *t, size_t cap) { for (size_t i = 0; i < cap && t[i]; i++) if (!strchr("ACGT", t[i])) return false; return true; };
    for (int i = 0; i < m->par.n_adapter; i++)
        if (!acgt(m->par.adapter[i], 63)) { bsx_set_error("packed read input needs upper-case ACGT adapters (got %s)", m->par.adapter[i]); return BSX_ERR_UNSUPPORTED; }
    if (m->par.rrbs && !acgt(m->par.digest_site, sizeof m->par.digest_site)) { bsx_set_error("packed read input needs an upper-case ACGT digestion site"); return BSX_ERR_UNSUPPORTED; }
    if (m->meth) { bsx_set_error("packed read input cannot feed the attached methylation pile-up (it reads the ASCII bases)"); return BSX_ERR_UNSUPPORTED; }
    return BSX_OK;
}

static int upload_slot(bsx_mapper *m, int si, uint32_t n, const char *sa, const uint16_t *la, const char *sb, const uint16_t *lb, cudaStream_t st,
                       bool packed = false) {
    bsx_slot &s = m->slot[si];
    if (n > m->max_batch) { bsx_set_error("batch of %u reads exceeds max_batch %u", n, m->max_batch); return BSX_ERR_ARG; }
    const size_t slot_bytes = packed ? bsx_packed_stride(m->stride) : (size_t)m->stride;
    s.packed = packed;
    BSX_CUDA_CHECK(cudaMemcpyAsync(s.d_seq_a, sa, (size_t)n * slot_bytes, cudaMemcpyHostToDevice, st));
    BSX_CUDA_CHECK(cudaMemcpyAsync(s.d_len_a, la, (size_t)n * 2, cudaMemcpyHostToDevice, st));
    if (sb) {
        int rc = alloc_pe(m); if (rc) return rc;
        BSX_CUDA_CHECK(cudaMemcpyAsync(s.d_seq_b, sb, (size_t)n * slot_bytes, cudaMemcpyHostToDevice, st));
        BSX_CUDA_CHECK(cudaMemcpyAsync(s.d_len_b, lb, (size_t)n * 2, cudaMemcpyHostToDevice, st));
    }
    return BSX_OK;
}

static int run_slot(bsx_mapper *m, int si, uint32_t n, uint32_t first_index, int readset, bool pe, cudaStream_t st) {
    bsx_slot &s = m->slot[si];
    if (n == 0) return BSX_OK;
    if (pe) { int rc = alloc_pe(m); if (rc) return rc; }
    const map_launch &k = pe ? m->pe : m->se;
    MapArgs a = m->base;
    a.seq_a = s.d_seq_a; a.len_a = s.d_len_a; a.seq_b = s.d_seq_b; a.len_b = s.d_len_b;
    a.n = n; a.first_index = first_index; a.readset = readset;
    a.out_a = s.d_out_a; a.out_b = s.d_out_b; a.out_pair = s.d_out_pair; a.cnt_a = s.d_cnt_a; a.cnt_b = s.d_cnt_b;
    a.work_counter = s.d_counter; a.hit_scratch = s.d_hits; a.dd_scratch = s.d_dd; a.pair_scratch = s.d_pairs;
    a.prep = s.d_prep; a.mates = pe ? 2 : 1;
    if (s.packed) { a.packed = 1; a.pk_maxlen = m->stride; a.pk_mask_off = (m->stride + 3) / 4; a.stride = (uint32_t)bsx_packed_stride(m->stride); }
    {   // 32 units per warp and atomic when the batch is large (>= 2 blocks per resident warp: the prepare phase runs
        // with all lanes busy); small batches take smaller blocks (>= 8 per warp) because there the tail decides --
        // config 5's 200 k heavy reads: 0.62 M reads/s with blocks of 32, 0.86 M with blocks of 4
        const uint64_t units = (uint64_t)n * (uint64_t)a.mates, warps = (uint64_t)(k.n_ctas * k.warps);
        const uint64_t want = units >= (1u << 19) ? 2 : 8;
        uint32_t b = 32;
        while (b > 4 && units / b < want * warps) b >>= 1;
        a.block_units = b;
    }
    if (pe) a.hit_stride = ((uint32_t)m->par.max_snp_num + 1) * 2 * ((uint32_t)m->par.max_num_hits + 1);
    BSX_CUDA_CHECK(cudaMemsetAsync(s.d_counter, 0, 4, st));
    m->launches++;
    int rc = launch_map(k, a, st);
    if (rc == BSX_OK && m->meth && !s.packed) {
        rc = bsx_meth_pile_mapped(m->meth, &m->meth_opts, m->meth_sam, m->par.report_repeat_hits, n, pe ? 2 : 1, readset, m->stride,
                                  s.d_seq_a, s.d_seq_b, s.d_out_a, s.d_out_b, s.d_out_pair, st);
        m->launches++;
    }
    return rc;
}

extern "C" int bsx_mapper_attach_meth(bsx_mapper *m, bsx_meth *meth, const bsx_meth_opts *o, int sam_rules) {
    if (!m || (meth && !o)) { bsx_set_error("bsx_mapper_attach_meth: bad argument"); return BSX_ERR_ARG; }
    if (meth && o->rm_dup && m->par.pairend && !sam_rules) {
        // methratio.py reads the paired file, then the unpaired one: its -r order is not the order the batches are mapped in
        bsx_set_error("-r (remove duplicates) with paired-end BSP output follows the order of two files: run methratio on them instead");
        return BSX_ERR_UNSUPPORTED;
    }
    m->meth = meth; m->meth_sam = sam_rules;
    if (o) m->meth_opts = *o;
    return BSX_OK;
}

static int download_slot(bsx_mapper *m, int si, uint32_t n, bool pe, bsx_pair_rec *op, bsx_rec *oa, bsx_rec *ob,
                         uint16_t *ca, uint16_t *cb, cudaStream_t st) {
    bsx_slot &s = m->slot[si];
    if (n == 0) return BSX_OK;
    if (oa) BSX_CUDA_CHECK(cudaMemcpyAsync(oa, s.d_out_a, (size_t)n * sizeof(bsx_rec), cudaMemcpyDeviceToHost, st));
    if (ca) BSX_CUDA_CHECK(cudaMemcpyAsync(ca, s.d_cnt_a, (size_t)n * 32, cudaMemcpyDeviceToHost, st));
    if (pe) {
        if (op) BSX_CUDA_CHECK(cudaMemcpyAsync(op, s.d_out_pair, (size_t)n * sizeof(bsx_pair_rec), cudaMemcpyDeviceToHost, st));
        if (ob) BSX_CUDA_CHECK(cudaMemcpyAsync(ob, s.d_out_b, (size_t)n * sizeof(bsx_rec), cudaMemcpyDeviceToHost, st));
        if (cb) BSX_CUDA_CHECK(cudaMemcpyAsync(cb, s.d_cnt_b, (size_t)n * 32, cudaMemcpyDeviceToHost, st));
    }
    return BSX_OK;
}

extern "C" int bsx_batch_upload(bsx_mapper *m, uint32_t n, const char *sa, const uint16_t *la, const char *sb, const uint16_t *lb, void *stream) {
    if (!m || !sa || !la) return BSX_ERR_ARG;
    BSX_CUDA_CHECK(cudaSetDevice(m->device));
    return upload_slot(m, 0, n, sa, la, sb, lb, pick_stream(m, 0, stream));
}
extern "C" int bsx_batch_upload_packed(bsx_mapper *m, uint32_t n, const uint8_t *sa, const uint16_t *la, const uint8_t *sb, const uint16_t *lb, void *stream) {
    if (!m || !sa || !la) return BSX_ERR_ARG;
    int rc = check_packed_ok(m); if (rc) return rc;
    BSX_CUDA_CHECK(cudaSetDevice(m->device));
    return upload_slot(m, 0, n, (const char *)sa, la, (const char *)sb, lb, pick_stream(m, 0, stream), true);
}
extern "C" int bsx_batch_run_se(bsx_mapper *m, uint32_t n, uint32_t first_index, int readset, void *stream) {
    if (!m) return BSX_ERR_ARG;
    BSX_CUDA_CHECK(cudaSetDevice(m->device));
    return run_slot(m, 0, n, first_index, readset, false, pick_stream(m, 0, stream));
}
extern "C" int bsx_batch_run_pe(bsx_mapper *m, uint32_t n, uint32_t first_index, void *stream) {
    if (!m) return BSX_ERR_ARG;
    BSX_CUDA_CHECK(cudaSetDevice(m->device));
    return run_slot(m, 0, n, first_index, 0, true, pick_stream(m, 0, stream));
}
extern "C" int bsx_batch_download_se(bsx_mapper *m, uint32_t n, bsx_rec *out, uint16_t *counts, void *stream) {
    if (!m) return BSX_ERR_ARG;
    BSX_CUDA_CHECK(cudaSetDevice(m->device));
    cudaStream_t st = pick_stream(m, 0, stream);
    int rc = download_slot(m, 0, n, false, nullptr, out, nullptr, counts, nullptr, st); if (rc) return rc;
    BSX_CUDA_CHECK(cudaStreamSynchronize(st));
    return BSX_OK;
}
extern "C" int bsx_batch_download_pe(bsx_mapper *m, uint32_t n, bsx_pair_rec *out, bsx_rec *oa, bsx_rec *ob, uint16_t *ca, uint16_t *cb, void *stream) {
    if (!m) return BSX_ERR_ARG;
    BSX_CUDA_CHECK(cudaSetDevice(m->device));
    cudaStream_t st = pick_stream(m, 0, stream);
    int rc = download_slot(m, 0, n, true, out, oa, ob, ca, cb, st); if (rc) return rc;
    BSX_CUDA_CHECK(cudaStreamSynchronize(st));
    return BSX_OK;
}
extern "C" int bsx_mapper_sync(bsx_mapper *m) {
    if (!m) return BSX_ERR_ARG;
    BSX_CUDA_CHECK(cudaSetDevice(m->device));
    BSX_CUDA_CHECK(cudaStreamSynchronize(m->slot[0].stream));
    BSX_CUDA_CHECK(cudaStreamSynchronize(m->slot[1].stream));
    return BSX_OK;
}

// Do_Batch with host buffers: sub-batches alternate between two slots/streams so the H2D copy of
// batch k+1 and the D2H copy of batch k-1 overlap the kernel of batch k (host buffers should be
// pinned for the overlap to be real).
static int map_host(bsx_mapper *m, bool pe, uint32_t n, const char *sa, const uint16_t *la, const char *sb, const uint16_t *lb,
                    uint32_t first_index, int readset, bsx_pair_rec *op, bsx_rec *oa, bsx_rec *ob, uint16_t *ca, uint16_t *cb,
                    bool packed = false) {
    BSX_CUDA_CHECK(cudaSetDevice(m->device));
    const size_t slot_bytes = packed ? bsx_packed_stride(m->stride) : (size_t)m->stride;
    uint32_t done = 0; int k = 0;
    while (done < n) {
        const int si = k & 1;
        cudaStream_t st = m->slot[si].stream;
        // the first sub-batch is small: its upload is the one copy no kernel hides
        const uint32_t nb = std::min(k == 0 && n > m->max_batch ? std::max(m->max_batch / 8u, 1u) : m->max_batch, n - done);
        BSX_CUDA_CHECK(cudaStreamSynchronize(st));    // slot free again
        int rc = upload_slot(m, si, nb, sa + (size_t)done * slot_bytes, la + done, sb ? sb + (size_t)done * slot_bytes : nullptr,
                             lb ? lb + done : nullptr, st, packed);
        if (rc) return rc;
        rc = run_slot(m, si, nb, first_index + done, readset, pe, st); if (rc) return rc;
        rc = download_slot(m, si, nb, pe, op ? op + done : nullptr, oa ? oa + done : nullptr, ob ? ob + done : nullptr,
                           ca ? ca + (size_t)done * 16 : nullptr, cb ? cb + (size_t)done * 16 : nullptr, st);
        if (rc) return rc;
        done += nb; k++;
    }
    BSX_CUDA_CHECK(cudaStreamSynchronize(m->slot[0].stream));
    BSX_CUDA_CHECK(cudaStreamSynchronize(m->slot[1].stream));
    return BSX_OK;
}

extern "C" int bsx_map_se(bsx_mapper *m, uint32_t n, const char *seqs, const uint16_t *lens, uint32_t first_index, int readset,
                          bsx_rec *out, uint16_t *counts) {
    if (m && n == 0) return BSX_OK;
    if (!m || !seqs || !lens || !out) { bsx_set_error("bsx_map_se: bad argument"); return BSX_ERR_ARG; }
    return map_host(m, false, n, seqs, lens, nullptr, nullptr, first_index, readset, nullptr, out, nullptr, counts, nullptr);
}
extern "C" int bsx_map_pe(bsx_mapper *m, uint32_t n, const char *sa, const uint16_t *la, const char *sb, const uint16_t *lb,
                          uint32_t first_index, bsx_pair_rec *out, bsx_rec *oa, bsx_rec *ob, uint16_t *ca, uint16_t *cb) {
    if (m && n == 0) return BSX_OK;
    if (!m || !sa || !la || !sb || !lb || !out || !oa || !ob) { bsx_set_error("bsx_map_pe: bad argument"); return BSX_ERR_ARG; }
    return map_host(m, true, n, sa, la, sb, lb, first_index, 0, out, oa, ob, ca, cb);
}

extern "C" int bsx_map_se_packed(bsx_mapper *m, uint32_t n, const uint8_t *packed, const uint16_t *lens, uint32_t first_index, int readset,
                                 bsx_rec *out, uint16_t *counts) {
    if (m && n == 0) return BSX_OK;
    if (!m || !packed || !lens || !out) { bsx_set_error("bsx_map_se_packed: bad argument"); return BSX_ERR_ARG; }
    int rc = check_packed_ok(m); if (rc) return rc;
    return map_host(m, false, n, (const char *)packed, lens, nullptr, nullptr, first_index, readset, nullptr, out, nullptr, counts, nullptr, true);
}
extern "C" int bsx_map_pe_packed(bsx_mapper *m, uint32_t n, const uint8_t *pa, const uint16_t *la, const uint8_t *pb, const uint16_t *lb,
                                 uint32_t first_index, bsx_pair_rec *out, bsx_rec *oa, bsx_rec *ob, uint16_t *ca, uint16_t *cb) {
    if (m && n == 0) return BSX_OK;
    if (!m || !pa || !la || !pb || !lb || !out || !oa || !ob) { bsx_set_error("bsx_map_pe_packed: bad argument"); return BSX_ERR_ARG; }
    int rc = check_packed_ok(m); if (rc) return rc;
    return map_host(m, true, n, (const char *)pa, la, (const char *)pb, lb, first_index, 0, out, oa, ob, ca, cb, true);
}

extern "C" int bsx_mapper_stats(bsx_mapper *m, bsx_stats *out, int reset) {
    if (!m || !out) return BSX_ERR_ARG;
    BSX_CUDA_CHECK(cudaSetDevice(m->device));
    BSX_CUDA_CHECK(cudaDeviceSynchronize());
    BSX_CUDA_CHECK(cudaMemcpy(out, m->d_stats, sizeof(bsx_stats), cudaMemcpyDeviceToHost));
    if (reset) BSX_CUDA_CHECK(cudaMemset(m->d_stats, 0, sizeof(bsx_stats)));
    return BSX_OK;
}
extern "C" uint64_t bsx_mapper_launches(const bsx_mapper *m) { return m ? m->launches : 0; }

// test hook: seed-selection state of the last SE batch (BSX_DEBUG_SEEDS=1), 40 u32 per read
extern "C" int bsx_mapper_debug_seeds(bsx_mapper *m, uint32_t n, uint32_t *dst) {
    if (!m || !m->d_debug) { bsx_set_error("debug buffer not enabled (set BSX_DEBUG_SEEDS=1 before bsx_mapper_create)"); return BSX_ERR_ARG; }
    BSX_CUDA_CHECK(cudaMemcpy(dst, m->d_debug, (size_t)n * 40 * 4, cudaMemcpyDeviceToHost));
    return BSX_OK;
}
