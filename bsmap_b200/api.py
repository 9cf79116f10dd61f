"""Python mirror of the reference's RefSeq / SingleAlign / PairAlign seam over the C ABI."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import lib as _l
from .lib import CONV_BINS, CT_SNP_MODES, MBIAS_CYCLES, METH_READ2, PAIR_REC, REC, BsxError, IndexInfo, MethOpts, Params, Stats, check, load, strs


def make_params(s=16, I=4, v=2, w=1000, r=1, m=28, x=500, n=0, pairend=0, S=0, f=5, L=144,
                out_sam=1, u=0, R=0, D=None, A=()) -> Params:
    """Param defaults (param.cpp:6-83) + the side effects of mGetOptions (main.cpp:234-289):
    -D forces seed 12 / interval 1 whatever -s / -I say (App. B Q17)."""
    p = Params()
    p.seed_size, p.index_interval, p.max_snp_num, p.max_num_hits = s, I, v, w
    p.report_repeat_hits, p.min_insert, p.max_insert, p.chains = r, m, x, n
    p.pairend, p.randseed, p.max_ns, p.max_readlen = pairend, S, f, L
    p.out_sam, p.out_unmap, p.out_ref = out_sam, u, R
    if D:
        if "-" not in D:
            raise ValueError("Digestion position not marked, use '-' to mark. example: 'C-CGG'")
        p.digest_pos = D.index("-")
        p.digest_site = D.replace("-", "").encode()
        p.rrbs, p.index_interval, p.seed_size = 1, 1, 12
    if len(A) > 10:
        raise ValueError("at most 10 adapters")
    p.n_adapter = len(A)
    for i, a in enumerate(A):
        p.adapter[i].value = a.encode()[:63]
    return p


def pack_reads(seqs, stride=None):
    """list of bytes -> (uint8[n, stride] zero padded, uint16 lens); stride is a multiple of 16"""
    n = len(seqs)
    lens = np.array([min(len(s), 65535) for s in seqs], dtype=np.uint16)
    need = int(lens.max()) if n else 16
    stride = stride or max(16, (min(need, 160) + 15) // 16 * 16)
    buf = np.zeros((n, stride), dtype=np.uint8)
    for i, s in enumerate(seqs):
        k = min(len(s), stride)
        buf[i, :k] = np.frombuffer(s[:k], dtype=np.uint8)
    return buf, lens


def pack_reads_2bit(buf: np.ndarray, lens: np.ndarray, threads: int = 0):
    """ASCII read slots -> packed slots (2-bit bases + valid mask, bsx_packed_stride bytes each) -> (packed, lower-case bases met)"""
    n, stride = buf.shape
    ps = int(load().bsx_packed_stride(stride))
    out = np.empty((n, ps), dtype=np.uint8)
    low = C.c_uint64(0)
    check(load().bsx_pack_reads(n, buf.ctypes.data, stride, lens.ctypes.data, out.ctypes.data, C.byref(low), threads))
    return out, int(low.value)


def _ptr(a):
    return a.ctypes.data if a is not None else None


class Index:
    """RefSeq: 2-bit packed Watson/Crick strands + bisulfite seed table, resident on one GPU."""

    def __init__(self, params: Params, names, seqs, device: int = 0, _handle=None):
        self.p = params
        self.device = device
        if _handle is not None:
            self.h = _handle
            return
        L = load()
        self._keep = [s if isinstance(s, bytes) else (s.tobytes() if isinstance(s, np.ndarray) else bytes(s)) for s in seqs]
        lens = np.array([len(s) for s in self._keep], dtype=np.uint32)
        h = C.c_void_p()
        check(L.bsx_index_create(C.byref(params), len(names), strs(names), strs(self._keep), lens.ctypes.data, device, C.byref(h)))
        self.h = h
        self._keep = None

    @classmethod
    def from_fasta(cls, params: Params, path: str, device: int = 0):
        h = C.c_void_p()
        check(load().bsx_index_create_from_fasta(C.byref(params), path.encode(), device, C.byref(h)))
        return cls(params, None, None, device, _handle=h)

    @classmethod
    def from_pointers(cls, params: Params, names, ptrs, lens, device: int = 0):
        """sequences already in host memory at raw addresses (bench: pinned torch tensors)"""
        arr = (C.c_char_p * len(names))()
        for i, a in enumerate(ptrs):
            arr[i] = C.cast(C.c_void_p(int(a)), C.c_char_p)
        ln = np.asarray(lens, dtype=np.uint32)
        h = C.c_void_p()
        check(load().bsx_index_create(C.byref(params), len(names), strs(names), arr, ln.ctypes.data, device, C.byref(h)))
        return cls(params, None, None, device, _handle=h)

    @classmethod
    def text_only(cls, params: Params, names, seqs):
        """host-only index for the text layer (format_*); cannot map"""
        keep = [s if isinstance(s, bytes) else bytes(s) for s in seqs]
        lens = np.array([len(s) for s in keep], dtype=np.uint32)
        h = C.c_void_p()
        check(load().bsx_index_create_text_only(C.byref(params), len(names), strs(names), strs(keep), lens.ctypes.data, C.byref(h)))
        return cls(params, None, None, -1, _handle=h)

    @classmethod
    def text_only_from_fasta(cls, params: Params, path: str):
        h = C.c_void_p()
        check(load().bsx_index_create_text_only_from_fasta(C.byref(params), os.fsencode(path), C.byref(h)))
        return cls(params, None, None, -1, _handle=h)

    def save_packed(self, path: str):
        """packed reference cache: forward strand, blocks, names, sizes (WGBS; independent of -s / -I)"""
        check(load().bsx_index_save_packed(self.h, os.fsencode(path)))

    @classmethod
    def from_packed(cls, params: Params, path: str, device: int = 0):
        h = C.c_void_p()
        check(load().bsx_index_create_from_packed(C.byref(params), os.fsencode(path), device, C.byref(h)))
        return cls(params, None, None, device, _handle=h)

    @classmethod
    def packed(cls, names, seqs, device: int = 0):
        """packed reference only (no seed table): enough for Meth, cannot map"""
        keep = [s if isinstance(s, bytes) else bytes(s) for s in seqs]
        lens = np.array([len(s) for s in keep], dtype=np.uint32)
        h = C.c_void_p()
        check(load().bsx_index_create_packed(len(names), strs(names), strs(keep), lens.ctypes.data, device, C.byref(h)))
        return cls(make_params(), None, None, device, _handle=h)

    def replicate(self, device: int) -> "Index":
        """full replica on another GPU over NVLink (cudaMemcpyPeer): the one-time index broadcast"""
        h = C.c_void_p()
        check(load().bsx_index_replicate(self.h, device, C.byref(h)))
        return Index(self.p, None, None, device, _handle=h)

    def meta(self) -> bytes:
        n = load().bsx_index_meta_size(self.h)
        b = C.create_string_buffer(n)
        check(load().bsx_index_meta_export(self.h, b, n))
        return b.raw

    @classmethod
    def shell(cls, params: Params, meta: bytes, device: int) -> "Index":
        h = C.c_void_p()
        check(load().bsx_index_create_shell(meta, len(meta), device, C.byref(h)))
        return cls(params, None, None, device, _handle=h)

    def device_buffers(self):
        ptrs = (C.c_void_p * 8)()
        sizes = (C.c_size_t * 8)()
        n = load().bsx_index_device_buffers(self.h, ptrs, sizes, 8)
        return [(int(ptrs[i] or 0), int(sizes[i])) for i in range(n)]

    @property
    def info(self) -> IndexInfo:
        i = IndexInfo()
        check(load().bsx_index_get_info(self.h, C.byref(i)))
        return i

    def names(self):
        return [load().bsx_index_seq_name(self.h, k).decode() for k in range(self.info.n_seq)]

    def download(self, what: str) -> np.ndarray:
        i = self.info
        which = {"refcat": (0, i.n_words), "crefcat": (1, i.n_words), "anchor": (2, i.n_seq + 1),
                 "tab": (3, i.n_tab), "pos": (4, i.n_entries), "tag": (5, i.n_entries),
                 "ctx": (6, i.ctx_words * i.n_entries)}[what]
        out = np.empty(int(which[1]), dtype=np.uint32)
        check(load().bsx_index_download(self.h, which[0], out.ctypes.data, out.nbytes))
        return out

    def header(self) -> bytes:
        n = load().bsx_format_header(self.h, None, 0)
        b = C.create_string_buffer(n + 1)
        load().bsx_format_header(self.h, b, n + 1)
        return b.raw[:n]

    def close(self):
        if getattr(self, "h", None) and _l._lib is not None:
            _l._lib.bsx_index_destroy(self.h)
        self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Mapper:
    """SingleAlign / PairAlign: ImportBatchReads + Do_Batch on the device."""

    def __init__(self, index: Index, params: Params = None, max_batch: int = 1 << 20, stride: int = 160):
        self.index = index
        self.p = params or index.p
        self.max_batch, self.stride = max_batch, stride
        h = C.c_void_p()
        check(load().bsx_mapper_create(index.h, C.byref(self.p), max_batch, stride, C.byref(h)))
        self.h = h

    # --- Do_Batch with host buffers (end to end) ---
    def map_se(self, buf: np.ndarray, lens: np.ndarray, first_index=0, readset=0, want_counts=True):
        n = len(lens)
        assert buf.shape[1] == self.stride and buf.dtype == np.uint8 and buf.flags.c_contiguous
        out = np.zeros(n, dtype=REC)
        counts = np.zeros((n, 16), dtype=np.uint16) if want_counts else None
        check(load().bsx_map_se(self.h, n, buf.ctypes.data, lens.ctypes.data, first_index, readset, out.ctypes.data, _ptr(counts)))
        return out, counts

    def map_se_packed(self, packed: np.ndarray, lens: np.ndarray, first_index=0, readset=0, want_counts=True):
        """Do_Batch on packed read slots (pack_reads_2bit of slots with this mapper's stride)"""
        n = len(lens)
        assert packed.dtype == np.uint8 and packed.flags.c_contiguous and packed.shape[1] == load().bsx_packed_stride(self.stride)
        out = np.zeros(n, dtype=REC)
        counts = np.zeros((n, 16), dtype=np.uint16) if want_counts else None
        check(load().bsx_map_se_packed(self.h, n, packed.ctypes.data, lens.ctypes.data, first_index, readset, out.ctypes.data, _ptr(counts)))
        return out, counts

    def map_se_packed_ptr(self, n, packed_ptr, len_ptr, out_ptr, counts_ptr=None, first_index=0, readset=0):
        check(load().bsx_map_se_packed(self.h, n, packed_ptr, len_ptr, first_index, readset, out_ptr, counts_ptr))

    def map_pe_packed(self, pk_a, lens_a, pk_b, lens_b, first_index=0):
        n = len(lens_a)
        pr = np.zeros(n, dtype=PAIR_REC)
        ra, rb = np.zeros(n, dtype=REC), np.zeros(n, dtype=REC)
        ca, cb = np.zeros((n, 16), dtype=np.uint16), np.zeros((n, 16), dtype=np.uint16)
        check(load().bsx_map_pe_packed(self.h, n, pk_a.ctypes.data, lens_a.ctypes.data, pk_b.ctypes.data, lens_b.ctypes.data,
                                       first_index, pr.ctypes.data, ra.ctypes.data, rb.ctypes.data, ca.ctypes.data, cb.ctypes.data))
        return pr, ra, rb, ca, cb

    def upload_packed(self, n, packed_ptr, len_ptr, packed_b_ptr=None, len_b_ptr=None, stream=None):
        check(load().bsx_batch_upload_packed(self.h, n, packed_ptr, len_ptr, packed_b_ptr, len_b_ptr, stream))

    def map_se_ptr(self, n, seq_ptr, len_ptr, out_ptr, counts_ptr=None, first_index=0, readset=0):
        """raw-address form (pinned host buffers owned by the caller)"""
        check(load().bsx_map_se(self.h, n, seq_ptr, len_ptr, first_index, readset, out_ptr, counts_ptr))

    def map_pe(self, buf_a, lens_a, buf_b, lens_b, first_index=0):
        n = len(lens_a)
        assert buf_a.shape[1] == self.stride and buf_b.shape[1] == self.stride
        pr = np.zeros(n, dtype=PAIR_REC)
        ra, rb = np.zeros(n, dtype=REC), np.zeros(n, dtype=REC)
        ca, cb = np.zeros((n, 16), dtype=np.uint16), np.zeros((n, 16), dtype=np.uint16)
        check(load().bsx_map_pe(self.h, n, buf_a.ctypes.data, lens_a.ctypes.data, buf_b.ctypes.data, lens_b.ctypes.data,
                                first_index, pr.ctypes.data, ra.ctypes.data, rb.ctypes.data, ca.ctypes.data, cb.ctypes.data))
        return pr, ra, rb, ca, cb

    def map_pe_ptr(self, n, seq_a_ptr, len_a_ptr, seq_b_ptr, len_b_ptr, pair_ptr, out_a_ptr, out_b_ptr, cnt_a_ptr=None, cnt_b_ptr=None, first_index=0):
        """raw-address form (pinned host buffers owned by the caller)"""
        check(load().bsx_map_pe(self.h, n, seq_a_ptr, len_a_ptr, seq_b_ptr, len_b_ptr, first_index, pair_ptr, out_a_ptr, out_b_ptr, cnt_a_ptr, cnt_b_ptr))

    # --- staged form: inputs resident in HBM ---
    def upload(self, n, seq_ptr, len_ptr, seq_b_ptr=None, len_b_ptr=None, stream=None):
        check(load().bsx_batch_upload(self.h, n, seq_ptr, len_ptr, seq_b_ptr, len_b_ptr, stream))

    def run_se(self, n, first_index=0, readset=0, stream=None):
        check(load().bsx_batch_run_se(self.h, n, first_index, readset, stream))

    def run_pe(self, n, first_index=0, stream=None):
        check(load().bsx_batch_run_pe(self.h, n, first_index, stream))

    def download_se(self, n, want_counts=False, stream=None):
        out = np.zeros(n, dtype=REC)
        counts = np.zeros((n, 16), dtype=np.uint16) if want_counts else None
        check(load().bsx_batch_download_se(self.h, n, out.ctypes.data, _ptr(counts), stream))
        return out, counts

    def sync(self):
        check(load().bsx_mapper_sync(self.h))

    def stats(self, reset=False) -> dict:
        s = Stats()
        check(load().bsx_mapper_stats(self.h, C.byref(s), 1 if reset else 0))
        return s.as_dict()

    @property
    def launches(self) -> int:
        return int(load().bsx_mapper_launches(self.h))

    def debug_seeds(self, n):
        out = np.zeros((n, 40), dtype=np.uint32)
        check(load().bsx_mapper_debug_seeds(self.h, n, out.ctypes.data))
        return out

    # --- text (s_OutHit & co) ---
    def format_se(self, names, seqs, quals, recs, counts=None, readset=0):
        n = len(names)
        args = (self.index.h, C.byref(self.p), n, strs(names), strs(seqs), strs(quals), readset, recs.ctypes.data, _ptr(counts))
        na = C.c_uint32(0)
        need = load().bsx_format_se(*args, None, 0, C.byref(na))
        b = C.create_string_buffer(need + 1)
        load().bsx_format_se(*args, b, need + 1, C.byref(na))
        return b.raw[:need], na.value

    def format_pe(self, names_a, seqs_a, quals_a, names_b, seqs_b, quals_b, pr, ra, rb, ca=None, cb=None):
        n = len(names_a)
        args = (self.index.h, C.byref(self.p), n, strs(names_a), strs(seqs_a), strs(quals_a), strs(names_b), strs(seqs_b),
                strs(quals_b), pr.ctypes.data, ra.ctypes.data, rb.ctypes.data, _ptr(ca), _ptr(cb))
        nu = C.c_size_t(0)
        st = (C.c_uint32 * 3)()
        need = load().bsx_format_pe(*args, None, 0, None, 0, C.byref(nu), st)
        b, bu = C.create_string_buffer(need + 1), C.create_string_buffer(nu.value + 1)
        load().bsx_format_pe(*args, b, need + 1, bu, nu.value + 1, C.byref(nu), st)
        return b.raw[:need], bu.raw[:nu.value], tuple(st)

    def close(self):
        if getattr(self, "h", None) and _l._lib is not None:
            _l._lib.bsx_mapper_destroy(self.h)
        self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Reads:
    """One FASTA / FASTQ read file: ReadClass::CheckFile + LoadBatchReads (reads.cpp:13-119)."""

    def __init__(self, path: str, zero_qual: int = ord("!"), max_readlen: int = 144):
        h = C.c_void_p()
        check(load().bsx_reads_open(os.fsencode(path), zero_qual, max_readlen, C.byref(h)))
        self.h = h

    @property
    def kind(self) -> str:
        return {0: "fastq", 1: "fasta", 3: "bam"}[load().bsx_reads_kind(self.h)]

    @property
    def failed(self) -> bool:
        """a streamed input (gzip, pipe) ended in an error: corrupt or truncated data"""
        return bool(load().bsx_reads_failed(self.h))

    def set_readset(self, readset: int):
        """BAM input: 0 single-end, 1 / 2 = file a / b of a pair interleaved in one BAM"""
        load().bsx_reads_set_readset(self.h, readset)

    def skip(self, n_reads: int):
        load().bsx_reads_skip(self.h, n_reads)

    def force_token_reader(self, on: bool = True):
        load().bsx_reads_force_token_reader(self.h, int(on))

    def next(self, want: int, stride: int = 160, threads: int = 0):
        """load up to `want` reads -> (n, bases[n, stride] u8 zero padded, lens[n] u16)"""
        buf = np.empty((want, stride), dtype=np.uint8)
        lens = np.empty(want, dtype=np.uint16)
        n = load().bsx_reads_next(self.h, want, stride, buf.ctypes.data, lens.ctypes.data, threads)
        return n, buf[:n], lens[:n]

    def get(self, i: int):
        """(name, bases, qualities) of read i of the current batch"""
        ptr = [C.c_void_p() for _ in range(3)]
        ln = [C.c_uint32() for _ in range(3)]
        check(load().bsx_reads_get(self.h, i, C.byref(ptr[0]), C.byref(ln[0]), C.byref(ptr[1]), C.byref(ln[1]), C.byref(ptr[2]), C.byref(ln[2])))
        return tuple(C.string_at(q.value, l.value) if l.value else b"" for q, l in zip(ptr, ln))

    def close(self):
        if getattr(self, "h", None) and _l._lib is not None:
            _l._lib.bsx_reads_close(self.h)
        self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def emit_se(index: Index, params: Params, reads: Reads, n: int, recs, counts, fd: int, readset=0, threads=0):
    """format the current batch of `reads` on `threads` host threads and write it to fd -> (bytes, n_aligned)"""
    na = C.c_uint32(0)
    w = load().bsx_emit_se(index.h, C.byref(params), reads.h, n, readset, recs.ctypes.data, _ptr(counts), threads, fd, C.byref(na))
    return w, na.value


def emit_pe(index: Index, params: Params, a: Reads, b: Reads, n: int, pr, ra, rb, ca, cb, fd: int, fd_unpair: int = -1, threads=0):
    st = (C.c_uint32 * 3)()
    w = load().bsx_emit_pe(index.h, C.byref(params), a.h, b.h, n, pr.ctypes.data, ra.ctypes.data, rb.ctypes.data, _ptr(ca), _ptr(cb),
                           threads, fd, fd_unpair, st)
    return w, tuple(st)


def meth_opts(unique=False, pair=False, meth0=False, trim_fillin=2, combine_cpg=False, min_depth=1, rm_dup=False) -> MethOpts:
    return MethOpts(int(unique), int(pair), int(meth0), int(trim_fillin), int(combine_cpg), int(min_depth), int(rm_dup))


class Meth:
    """methratio.py's per-position counters on the device (bsx_meth_*)"""

    def __init__(self, index: Index, opts: MethOpts = None):
        self.index, self.o = index, opts or meth_opts()
        h = C.c_void_p()
        check(load().bsx_meth_create(index.h, C.byref(h)))
        self.h = h
        self.n_valid = 0

    def add(self, seqs, chr_idx, pos, strand, insert, mate_pos, flags, read2=None):
        """seqs: list of bytes (SEQ as printed); strand: bit 0 / 1 = first / second ZS character is '-';
        read2: optional per-alignment truth values (FLAG 0x80), setting BSX_METH_READ2 in flags"""
        n = len(seqs)
        longest = max((len(s) for s in seqs), default=0)
        if longest > 65535:                                  # the lengths bsx_meth_add takes are 16-bit
            raise ValueError("Meth.add: a SEQ of %d bases; at most 65535 are supported" % longest)
        if read2 is not None:
            flags = np.asarray(flags, dtype=np.uint8) | np.where(np.asarray(read2, dtype=bool), np.uint8(METH_READ2), np.uint8(0))
        buf, lens = pack_reads(seqs, stride=max(16, (max((len(s) for s in seqs), default=1) + 15) // 16 * 16))
        arr = lambda a, t: np.ascontiguousarray(np.asarray(a, dtype=t))
        c, p, st, ins, mt, fl = arr(chr_idx, np.uint32), arr(pos, np.uint32), arr(strand, np.uint8), arr(insert, np.int32), arr(mate_pos, np.int32), arr(flags, np.uint8)
        nv = C.c_uint64(0)
        check(load().bsx_meth_add(self.h, C.byref(self.o), n, buf.ctypes.data, buf.shape[1], lens.ctypes.data, c.ctypes.data, p.ctypes.data,
                                  st.ctypes.data, ins.ctypes.data, mt.ctypes.data, fl.ctypes.data, C.byref(nv)))
        self.n_valid = nv.value
        return nv.value

    def attach(self, mapper: "Mapper", sam_rules: bool = True):
        """pile up every batch `mapper` maps from now on, on the device, without SAM text in between"""
        check(load().bsx_mapper_attach_meth(mapper.h, self.h, C.byref(self.o), int(sam_rules)))

    def valid(self) -> int:
        nv = C.c_uint64(0)
        check(load().bsx_meth_valid_count(self.h, C.byref(nv)))
        self.n_valid = nv.value
        return nv.value

    def counters(self, k: int):
        """(meth, depth) of reference sequence k"""
        n = load().bsx_index_seq_size(self.index.h, k)
        m, d = np.zeros(n, dtype=np.uint32), np.zeros(n, dtype=np.uint32)
        check(load().bsx_meth_download(self.h, C.byref(self.o), k, m.ctypes.data, d.ctypes.data))
        return m, d

    def enable_mbias(self):
        """track the M-bias (methylation by read, C context and cycle); before the first add / mapped batch"""
        check(load().bsx_meth_enable_mbias(self.h))

    def set_ignore(self, r1_5p=0, r1_3p=0, r2_5p=0, r2_3p=0):
        """drop calls in the first / last cycles of read 1 / read 2 from the counters and the M-bias; before the first add"""
        v = (C.c_int32 * 4)(int(r1_5p), int(r1_3p), int(r2_5p), int(r2_3p))
        check(load().bsx_meth_set_ignore(self.h, v))

    def mbias(self):
        """-> (uint64 array [read][context CpG/CHG/CHH][cycle][methylated, unmethylated], calls past the last cycle)"""
        h = np.zeros((2, 3, MBIAS_CYCLES, 2), dtype=np.uint64)
        over = C.c_uint64(0)
        check(load().bsx_meth_mbias(self.h, h.ctypes.data, C.byref(over)))
        return h, over.value

    def write_mbias(self, fd: int) -> int:
        """the M-bias report (include/bsmap_b200.h) to fd; returns bytes written"""
        w = load().bsx_meth_write_mbias(self.h, fd)
        if w == 0:
            check(1)
        return w

    def enable_ct_snp(self, mode: str):
        """count C/T SNP evidence from the opposite strand and write the 12-column table; mode "no-action",
        "correct" or "skip" (include/bsmap_b200.h); before the first add / mapped batch"""
        if mode not in CT_SNP_MODES:
            raise ValueError("ct-snp mode must be one of %s, not %r" % (", ".join(CT_SNP_MODES), mode))
        check(load().bsx_meth_enable_ct_snp(self.h, CT_SNP_MODES[mode]))

    def ct_snp_counters(self, k: int):
        """(confirm, snp) evidence of reference sequence k, after -g combining"""
        n = load().bsx_index_seq_size(self.index.h, k)
        c, s = np.zeros(n, dtype=np.uint32), np.zeros(n, dtype=np.uint32)
        check(load().bsx_meth_download_ct_snp(self.h, C.byref(self.o), k, c.ctypes.data, s.ctypes.data))
        return c, s

    def enable_conversion_filter(self, threshold: int = 3):
        """score every alignment by its methylated non-CpG calls and drop those scoring `threshold` or more (0..255;
        0 only counts them), include/bsmap_b200.h; before the first add / mapped batch"""
        check(load().bsx_meth_enable_conversion_filter(self.h, int(threshold)))

    def conversion(self):
        """-> (uint64 array [CONV_BINS]: valid alignments by score, the last bin 255 or more; alignments dropped)"""
        h = np.zeros(CONV_BINS, dtype=np.uint64)
        dropped = C.c_uint64(0)
        check(load().bsx_meth_conversion(self.h, h.ctypes.data, C.byref(dropped)))
        return h, dropped.value

    def write_conversion(self, fd: int) -> int:
        """the conversion report (include/bsmap_b200.h) to fd; returns bytes written"""
        w = load().bsx_meth_write_conversion(self.h, fd)
        if w == 0:
            check(1)
        return w

    def enable_pdr(self, min_cpg: int = 4):
        """score every alignment by its CpG calls for the proportion of discordant reads: an alignment with `min_cpg`
        (1..255) or more CpG calls is concordant or discordant (include/bsmap_b200.h); before the first add / mapped batch"""
        check(load().bsx_meth_enable_pdr(self.h, int(min_cpg)))

    def pdr_counters(self, k: int):
        """(concordant, discordant) CpG calls of informative alignments on reference sequence k, after -g combining"""
        n = load().bsx_index_seq_size(self.index.h, k)
        c, d = np.zeros(n, dtype=np.uint32), np.zeros(n, dtype=np.uint32)
        check(load().bsx_meth_download_pdr(self.h, C.byref(self.o), k, c.ctypes.data, d.ctypes.data))
        return c, d

    def pdr(self):
        """-> (informative alignments, discordant alignments)"""
        inf, disc = C.c_uint64(0), C.c_uint64(0)
        check(load().bsx_meth_pdr(self.h, C.byref(inf), C.byref(disc)))
        return inf.value, disc.value

    def write_pdr(self, seqs, fd: int, chroms=None, threads=0) -> int:
        """the PDR file (include/bsmap_b200.h) to fd; seqs and chroms as in write; returns bytes written"""
        keep = [s if isinstance(s, bytes) else bytes(s) for s in seqs]
        lens = np.array([len(s) for s in keep], dtype=np.uint32)
        sel = None if chroms is None else np.ascontiguousarray(np.asarray(chroms, dtype=np.uint8))
        w = load().bsx_meth_write_pdr(self.h, C.byref(self.o), strs(keep), lens.ctypes.data, _ptr(sel), threads, fd)
        if w == 0:
            check(1)
        return w

    @staticmethod
    def _regions(chr_idx, start, end):
        arr = lambda a, t: np.ascontiguousarray(np.asarray(a, dtype=t).reshape(-1))
        c, s, e = arr(chr_idx, np.uint32), arr(start, np.uint64), arr(end, np.uint64)
        if not len(c) == len(s) == len(e):
            raise ValueError("chr_idx, start and end differ in length (%d, %d, %d)" % (len(c), len(s), len(e)))
        return c, s, e

    def regions(self, chr_idx, start, end) -> np.ndarray:
        """-> uint64 array [region][context CpG/CHG/CHH][sites, covered, C, CT] over the 0-based half-open regions
        (sequence chr_idx[r], start[r], end[r]); the rules are in include/bsmap_b200.h"""
        c, s, e = self._regions(chr_idx, start, end)
        out = np.zeros((len(c), 3, 4), dtype=np.uint64)
        check(load().bsx_meth_regions(self.h, C.byref(self.o), len(c), c.ctypes.data, s.ctypes.data, e.ctypes.data, out.ctypes.data))
        return out

    def regions_pdr(self, chr_idx, start, end):
        """-> (regions' array as in regions, uint64 array [region][concordant, discordant]: the sums over the PDR file's
        lines in each region); needs enable_pdr"""
        c, s, e = self._regions(chr_idx, start, end)
        out, pdr = np.zeros((len(c), 3, 4), dtype=np.uint64), np.zeros((len(c), 2), dtype=np.uint64)
        check(load().bsx_meth_regions_pdr(self.h, C.byref(self.o), len(c), c.ctypes.data, s.ctypes.data, e.ctypes.data, out.ctypes.data,
                                          pdr.ctypes.data))
        return out, pdr

    def write_regions(self, fd: int, chr_idx, start, end) -> int:
        """the region report (include/bsmap_b200.h) to fd; returns bytes written"""
        c, s, e = self._regions(chr_idx, start, end)
        w = load().bsx_meth_write_regions(self.h, C.byref(self.o), len(c), c.ctypes.data, s.ctypes.data, e.ctypes.data, fd)
        if w == 0:
            check(1)
        return w

    def write(self, seqs, fd: int, chroms=None, threads=0):
        keep = [s if isinstance(s, bytes) else bytes(s) for s in seqs]
        lens = np.array([len(s) for s in keep], dtype=np.uint32)
        sel = None if chroms is None else np.ascontiguousarray(np.asarray(chroms, dtype=np.uint8))
        st = (C.c_uint64 * 2)()
        w = load().bsx_meth_write(self.h, C.byref(self.o), strs(keep), lens.ctypes.data, _ptr(sel), threads, fd, st)
        return w, (st[0], st[1])

    def close(self):
        if getattr(self, "h", None) and _l._lib is not None:
            _l._lib.bsx_meth_destroy(self.h)
        self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def sam_to_sorted_bam(sam_path: str, bam_path: str, threads: int = 0):
    """SAM text -> coordinate-sorted BAM + .bai, the way `samtools view -bS | sort | index` (0.1.7) writes them"""
    check(load().bsx_sam_to_sorted_bam(os.fsencode(sam_path), os.fsencode(bam_path), threads))
