"""ctypes binding of libbsmap_b200.so (the C ABI declared in include/bsmap_b200.h).

There is no fallback: if the shared library is missing, or no CUDA device is usable, every entry
point raises.  Nothing here imports or calls the oracle.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("BSMAP_B200_LIB") or os.path.join(HERE, "libbsmap_b200.so")   # override: kernel A/B experiments

MAXSNPS, MAXHITS, MAX_READLEN = 15, 1000, 144


class BsxError(RuntimeError):
    pass


class Params(C.Structure):
    """bsx_params: the Param fields that reach the hot path (param.h:54-121)"""
    _fields_ = [(n, C.c_int32) for n in (
        "seed_size", "index_interval", "max_snp_num", "max_num_hits", "report_repeat_hits",
        "min_insert", "max_insert", "chains", "pairend", "rrbs", "randseed", "max_ns",
        "max_readlen", "out_sam", "out_unmap", "out_ref", "digest_pos", "n_adapter")] + [
        ("digest_site", C.c_char * 32), ("adapter", (C.c_char * 64) * 10)]


class IndexInfo(C.Structure):
    _fields_ = [("n_words", C.c_uint64), ("n_keys", C.c_uint64), ("n_entries", C.c_uint64),
                ("n_seq", C.c_uint32), ("device", C.c_int32), ("build_seconds", C.c_double), ("n_tab", C.c_uint64), ("ctx_words", C.c_uint32), ("pad_", C.c_uint32)]


class Stats(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("candidates", "probes", "overfetch", "full_extensions", "commits",
                                          "mapped", "list_entries", "gathers")]

    def as_dict(self):
        return {n: int(getattr(self, n)) for n, _ in self._fields_}


REC = np.dtype([("loc", "<u4"), ("chr", "<u4"), ("nhits", "<u4"), ("nm", "u1"), ("chain", "u1"),
                ("status", "u1"), ("len", "u1")])
PAIR_REC = np.dtype([("a_loc", "<u4"), ("a_chr", "<u4"), ("b_loc", "<u4"), ("b_chr", "<u4"),
                     ("insert", "<i4"), ("npairs", "<u4"), ("na", "u1"), ("nb", "u1"),
                     ("chain", "u1"), ("paired", "u1")])

class MethOpts(C.Structure):
    """bsx_meth_opts (include/bsmap_b200.h): methratio.py's options"""
    _fields_ = [(k, C.c_int32) for k in ("unique", "pair", "meth0", "trim_fillin", "combine_cpg", "min_depth", "rm_dup")]


EXPORTS = [
    "bsx_last_error", "bsx_device_count", "bsx_params_default", "bsx_index_create", "bsx_index_create_from_fasta",
    "bsx_index_create_text_only", "bsx_index_create_text_only_from_fasta", "bsx_index_destroy", "bsx_index_get_info", "bsx_index_seq_name", "bsx_index_seq_size", "bsx_index_download",
    "bsx_index_device_buffers", "bsx_index_replicate", "bsx_index_meta_size", "bsx_index_meta_export",
    "bsx_index_create_shell", "bsx_mapper_create", "bsx_mapper_destroy", "bsx_map_se", "bsx_map_pe",
    "bsx_batch_upload", "bsx_batch_run_se", "bsx_batch_run_pe", "bsx_batch_download_se", "bsx_batch_download_pe",
    "bsx_mapper_sync", "bsx_mapper_stats", "bsx_mapper_launches", "bsx_format_header", "bsx_format_se",
    "bsx_format_pe", "bsx_cli_main",
    "bsx_reads_open", "bsx_reads_close", "bsx_reads_kind", "bsx_reads_failed", "bsx_reads_skip", "bsx_reads_force_token_reader", "bsx_reads_set_readset",
    "bsx_reads_next", "bsx_reads_get", "bsx_emit_se", "bsx_emit_pe",
    "bsx_index_create_packed", "bsx_index_save_packed", "bsx_index_create_from_packed", "bsx_meth_opts_default", "bsx_meth_create", "bsx_meth_destroy", "bsx_meth_add", "bsx_meth_download",
    "bsx_meth_write", "bsx_methratio_main", "bsx_sam_to_sorted_bam", "bsx_mapper_attach_meth", "bsx_meth_valid_count",
    "bsx_packed_stride", "bsx_pack_reads", "bsx_map_se_packed", "bsx_map_pe_packed", "bsx_batch_upload_packed",
    "bsx_meth_enable_mbias", "bsx_meth_set_ignore", "bsx_meth_mbias", "bsx_meth_write_mbias",
    "bsx_meth_enable_ct_snp", "bsx_meth_download_ct_snp",
    "bsx_meth_enable_conversion_filter", "bsx_meth_conversion", "bsx_meth_write_conversion",
    "bsx_meth_regions", "bsx_meth_write_regions",
    "bsx_meth_enable_pdr", "bsx_meth_download_pdr", "bsx_meth_pdr", "bsx_meth_write_pdr", "bsx_meth_regions_pdr",
    "bsx_meth_enable_epialleles", "bsx_meth_cpg_sites", "bsx_meth_download_epialleles", "bsx_meth_epialleles", "bsx_meth_write_epialleles",
    "bsx_meth_enable_mhl", "bsx_meth_download_mhl", "bsx_meth_mhl", "bsx_meth_regions_mhl", "bsx_meth_write_mhl",
]

METH_READ2 = 8        # BSX_METH_READ2: alignment flag, read 2 (FLAG 0x80)
MBIAS_CYCLES = 512    # BSX_MBIAS_CYCLES
CONV_BINS = 256       # BSX_CONV_BINS
EPI_CPGS = 4          # BSX_EPI_CPGS
MHL_MAX_LEN = 16      # BSX_MHL_MAX_LEN
CT_SNP_MODES = {"no-action": 1, "correct": 2, "skip": 3}   # BSX_CT_SNP_*

_lib = None


def load():
    """dlopen the in-tree library; raises BsxError when it has not been built"""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise BsxError(f"{LIB_PATH} not found: build it with `python -m bsmap_b200.build` (no CPU fallback exists)")
    L = C.CDLL(LIB_PATH)
    vp, u32, i32, sz = C.c_void_p, C.c_uint32, C.c_int, C.c_size_t
    pp = C.POINTER(C.c_char_p)
    L.bsx_last_error.restype = C.c_char_p
    L.bsx_device_count.restype = i32
    L.bsx_params_default.argtypes = [C.POINTER(Params)]
    L.bsx_index_create.argtypes = [C.POINTER(Params), i32, pp, pp, vp, i32, C.POINTER(vp)]
    L.bsx_index_create_from_fasta.argtypes = [C.POINTER(Params), C.c_char_p, i32, C.POINTER(vp)]
    L.bsx_index_create_text_only.argtypes = [C.POINTER(Params), i32, pp, pp, vp, C.POINTER(vp)]
    L.bsx_index_create_text_only_from_fasta.argtypes = [C.POINTER(Params), C.c_char_p, C.POINTER(vp)]
    L.bsx_index_destroy.argtypes = [vp]
    L.bsx_index_get_info.argtypes = [vp, C.POINTER(IndexInfo)]
    L.bsx_index_seq_name.restype = C.c_char_p
    L.bsx_index_seq_name.argtypes = [vp, u32]
    L.bsx_index_seq_size.restype = u32
    L.bsx_index_seq_size.argtypes = [vp, u32]
    L.bsx_index_download.argtypes = [vp, i32, vp, sz]
    L.bsx_index_device_buffers.argtypes = [vp, C.POINTER(vp), C.POINTER(sz), i32]
    L.bsx_index_replicate.argtypes = [vp, i32, C.POINTER(vp)]
    L.bsx_index_meta_size.restype = sz
    L.bsx_index_meta_size.argtypes = [vp]
    L.bsx_index_meta_export.argtypes = [vp, vp, sz]
    L.bsx_index_create_shell.argtypes = [vp, sz, i32, C.POINTER(vp)]
    L.bsx_mapper_create.argtypes = [vp, C.POINTER(Params), u32, u32, C.POINTER(vp)]
    L.bsx_mapper_destroy.argtypes = [vp]
    L.bsx_map_se.argtypes = [vp, u32, vp, vp, u32, i32, vp, vp]
    L.bsx_map_pe.argtypes = [vp, u32, vp, vp, vp, vp, u32, vp, vp, vp, vp, vp]
    L.bsx_batch_upload.argtypes = [vp, u32, vp, vp, vp, vp, vp]
    L.bsx_batch_run_se.argtypes = [vp, u32, u32, i32, vp]
    L.bsx_batch_run_pe.argtypes = [vp, u32, u32, vp]
    L.bsx_batch_download_se.argtypes = [vp, u32, vp, vp, vp]
    L.bsx_batch_download_pe.argtypes = [vp, u32, vp, vp, vp, vp, vp, vp]
    L.bsx_mapper_sync.argtypes = [vp]
    L.bsx_mapper_stats.argtypes = [vp, C.POINTER(Stats), i32]
    L.bsx_mapper_launches.restype = C.c_uint64
    L.bsx_mapper_launches.argtypes = [vp]
    L.bsx_format_header.restype = sz
    L.bsx_format_header.argtypes = [vp, C.c_char_p, sz]
    L.bsx_format_se.restype = sz
    L.bsx_format_se.argtypes = [vp, C.POINTER(Params), u32, pp, pp, pp, i32, vp, vp, C.c_char_p, sz, C.POINTER(u32)]
    L.bsx_format_pe.restype = sz
    L.bsx_format_pe.argtypes = [vp, C.POINTER(Params), u32] + [pp] * 6 + [vp] * 5 + [
        C.c_char_p, sz, C.c_char_p, sz, C.POINTER(sz), C.POINTER(u32)]
    L.bsx_reads_open.argtypes = [C.c_char_p, i32, i32, C.POINTER(vp)]
    L.bsx_reads_close.argtypes = [vp]; L.bsx_reads_close.restype = None
    L.bsx_reads_kind.argtypes = [vp]
    L.bsx_reads_failed.argtypes = [vp]
    L.bsx_reads_skip.argtypes = [vp, C.c_uint64]; L.bsx_reads_skip.restype = None
    L.bsx_reads_set_readset.argtypes = [vp, i32]; L.bsx_reads_set_readset.restype = None
    L.bsx_reads_force_token_reader.argtypes = [vp, i32]; L.bsx_reads_force_token_reader.restype = None
    L.bsx_reads_next.argtypes = [vp, u32, u32, vp, vp, i32]; L.bsx_reads_next.restype = u32
    L.bsx_reads_get.argtypes = [vp, u32] + [C.POINTER(vp), C.POINTER(u32)] * 3
    L.bsx_emit_se.restype = sz
    L.bsx_emit_se.argtypes = [vp, C.POINTER(Params), vp, u32, i32, vp, vp, i32, i32, C.POINTER(u32)]
    L.bsx_emit_pe.restype = sz
    L.bsx_emit_pe.argtypes = [vp, C.POINTER(Params), vp, vp, u32] + [vp] * 5 + [i32, i32, i32, C.POINTER(u32)]
    L.bsx_index_save_packed.argtypes = [vp, C.c_char_p]
    L.bsx_index_create_from_packed.argtypes = [C.POINTER(Params), C.c_char_p, i32, C.POINTER(vp)]
    L.bsx_index_create_packed.argtypes = [i32, pp, pp, vp, i32, C.POINTER(vp)]
    L.bsx_meth_opts_default.argtypes = [C.POINTER(MethOpts)]; L.bsx_meth_opts_default.restype = None
    L.bsx_meth_create.argtypes = [vp, C.POINTER(vp)]
    L.bsx_meth_destroy.argtypes = [vp]
    L.bsx_meth_add.argtypes = [vp, C.POINTER(MethOpts), u32, vp, u32, vp, vp, vp, vp, vp, vp, vp, C.POINTER(C.c_uint64)]
    L.bsx_meth_download.argtypes = [vp, C.POINTER(MethOpts), u32, vp, vp]
    L.bsx_sam_to_sorted_bam.argtypes = [C.c_char_p, C.c_char_p, i32]
    L.bsx_mapper_attach_meth.argtypes = [vp, vp, C.POINTER(MethOpts), i32]
    L.bsx_meth_valid_count.argtypes = [vp, C.POINTER(C.c_uint64)]
    L.bsx_meth_write.restype = sz
    L.bsx_meth_write.argtypes = [vp, C.POINTER(MethOpts), pp, vp, vp, i32, i32, C.POINTER(C.c_uint64)]
    L.bsx_meth_enable_mbias.argtypes = [vp]
    L.bsx_meth_set_ignore.argtypes = [vp, C.POINTER(C.c_int32)]
    L.bsx_meth_mbias.argtypes = [vp, vp, C.POINTER(C.c_uint64)]
    L.bsx_meth_write_mbias.restype = sz
    L.bsx_meth_write_mbias.argtypes = [vp, i32]
    L.bsx_meth_enable_ct_snp.argtypes = [vp, i32]
    L.bsx_meth_download_ct_snp.argtypes = [vp, C.POINTER(MethOpts), u32, vp, vp]
    L.bsx_meth_enable_conversion_filter.argtypes = [vp, i32]
    L.bsx_meth_conversion.argtypes = [vp, vp, C.POINTER(C.c_uint64)]
    L.bsx_meth_write_conversion.restype = sz
    L.bsx_meth_write_conversion.argtypes = [vp, i32]
    L.bsx_meth_regions.argtypes = [vp, C.POINTER(MethOpts), C.c_uint64, vp, vp, vp, vp]
    L.bsx_meth_write_regions.restype = sz
    L.bsx_meth_write_regions.argtypes = [vp, C.POINTER(MethOpts), C.c_uint64, vp, vp, vp, i32]
    L.bsx_meth_enable_pdr.argtypes = [vp, i32]
    L.bsx_meth_download_pdr.argtypes = [vp, C.POINTER(MethOpts), u32, vp, vp]
    L.bsx_meth_pdr.argtypes = [vp, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    L.bsx_meth_write_pdr.restype = sz
    L.bsx_meth_write_pdr.argtypes = [vp, C.POINTER(MethOpts), pp, vp, vp, i32, i32]
    L.bsx_meth_regions_pdr.argtypes = [vp, C.POINTER(MethOpts), C.c_uint64, vp, vp, vp, vp, vp]
    L.bsx_meth_enable_epialleles.argtypes = [vp]
    L.bsx_meth_cpg_sites.argtypes = [vp, u32, C.POINTER(C.c_uint64)]
    L.bsx_meth_download_epialleles.argtypes = [vp, u32, vp, vp]
    L.bsx_meth_epialleles.argtypes = [vp, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    L.bsx_meth_write_epialleles.restype = sz
    L.bsx_meth_write_epialleles.argtypes = [vp, C.POINTER(MethOpts), pp, vp, vp, i32, i32]
    L.bsx_meth_enable_mhl.argtypes = [vp]
    L.bsx_meth_download_mhl.argtypes = [vp, u32, vp, vp]
    L.bsx_meth_mhl.argtypes = [vp, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    L.bsx_meth_regions_mhl.argtypes = [vp, C.POINTER(MethOpts), C.c_uint64, vp, vp, vp, vp, vp]
    L.bsx_meth_write_mhl.restype = sz
    L.bsx_meth_write_mhl.argtypes = [vp, C.POINTER(MethOpts), C.c_uint64, vp, vp, vp, i32]
    L.bsx_packed_stride.restype = sz
    L.bsx_packed_stride.argtypes = [u32]
    L.bsx_pack_reads.argtypes = [u32, vp, u32, vp, vp, C.POINTER(C.c_uint64), i32]
    L.bsx_map_se_packed.argtypes = [vp, u32, vp, vp, u32, i32, vp, vp]
    L.bsx_map_pe_packed.argtypes = [vp, u32, vp, vp, vp, vp, u32, vp, vp, vp, vp, vp]
    L.bsx_batch_upload_packed.argtypes = [vp, u32, vp, vp, vp, vp, vp]
    if hasattr(L, "bsx_mapper_debug_seeds"):
        L.bsx_mapper_debug_seeds.argtypes = [vp, u32, vp]
    _lib = L
    return L


def check(rc: int):
    if rc != 0:
        raise BsxError(f"bsmap_b200 error {rc}: {load().bsx_last_error().decode(errors='replace')}")


def strs(xs):
    arr = (C.c_char_p * len(xs))()
    arr[:] = [x if isinstance(x, bytes) else x.encode() for x in xs]
    return arr
