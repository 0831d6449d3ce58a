"""ctypes binding of libvarscot_scan.so (the C ABI declared in include/varscot_scan.h).

There is no Python or CPU fallback: importing this module without the built library raises, and every
compute entry point returns an error code (surfaced as VarscotError) when no sm_100 device is usable.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("VARSCOT_LIB") or os.path.join(_HERE, "libvarscot_scan.so")     # VARSCOT_LIB: a tuning build (tools/gpu_variants.sh)

VS_OK, VS_ERR_ARG, VS_ERR_CUDA, VS_ERR_NOMEM, VS_ERR_OVERFLOW, VS_ERR_NODEVICE, VS_ERR_IO = range(7)
GLEN = 23


class VarscotError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"varscot_scan error {code}: {msg}")
        self.code = code


class Hit(C.Structure):
    _fields_ = [("pos", C.c_uint32), ("info", C.c_uint32)]


class Record(C.Structure):
    _fields_ = [("guide", C.c_uint32), ("contig", C.c_uint32), ("pos", C.c_uint32),
                ("flag", C.c_uint16), ("mm", C.c_uint8), ("pad", C.c_uint8)]


class ScanStats(C.Structure):
    _fields_ = [("upload_ms", C.c_float), ("extract_ms", C.c_float), ("score_ms", C.c_float), ("total_ms", C.c_float),
                ("n_cand_fwd", C.c_uint64), ("n_cand_rev", C.c_uint64),
                ("n_blocks_fwd", C.c_uint64), ("n_blocks_rev", C.c_uint64),
                ("n_hits", C.c_uint64), ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64),
                ("launches", C.c_uint32), ("score_launches", C.c_uint32), ("n_chunks", C.c_uint32), ("redo_chunks", C.c_uint32),
                ("resolve_ms", C.c_float), ("index_reused", C.c_uint32), ("guide_passes", C.c_uint32), ("index_build_ms", C.c_float)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class LocHit(C.Structure):
    _fields_ = [("key", C.c_uint64), ("contig", C.c_uint32), ("info", C.c_uint32)]


HIT_SINK = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32)
RECORD_SINK = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32)
VS_OPT_KEEP_INDEX, VS_OPT_HIT_CAPACITY, VS_OPT_BUCKET_INDEX = 1, 2, 3


class TextView(C.Structure):
    _fields_ = [("n_bases", C.c_uint64), ("n_words", C.c_uint64), ("n_contigs", C.c_uint32), ("reserved", C.c_uint32),
                ("contig_off", C.c_void_p), ("bases", C.c_void_p), ("masks", C.c_void_p), ("sparse", C.c_void_p),
                ("n_sparse", C.c_uint64),
                ("em_code", C.c_void_p), ("em_dense", C.c_void_p), ("nm_runs", C.c_void_p), ("em_runs", C.c_void_p),
                ("n_nm_runs", C.c_uint64), ("n_em_runs", C.c_uint64)]


class MaskSource(C.Structure):
    _fields_ = [("em_code", C.c_void_p), ("em_dense", C.c_void_p), ("nm_runs", C.c_void_p), ("em_runs", C.c_void_p),
                ("n_nm_runs", C.c_uint64), ("n_em_runs", C.c_uint64), ("n_em_blocks", C.c_uint64)]


# every symbol include/varscot_scan.h declares (tests check the library exports all of them)
EXPORTS = [
    "vs_packer_new", "vs_packer_free", "vs_packer_append", "vs_packer_end_contig", "vs_packer_finish", "vs_pack_text", "vs_pack_text_planes",
    "vs_masks_from_planes", "vs_masks_sparse", "vs_mask_source_build", "vs_mask_source_free", "vs_text_save", "vs_text_load", "vs_text_masks", "vs_map_records", "vs_free", "vs_device_count",
    "vs_ctx_create", "vs_ctx_destroy", "vs_last_error", "vs_ctx_set_chunk_words", "vs_text_upload", "vs_host_alloc",
    "vs_host_free", "vs_host_register", "vs_host_unregister", "vs_ctx_set_option", "vs_index_drop", "vs_scan", "vs_scan_text", "vs_scan_fetch",
    "vs_scan_resolved", "vs_merge_resolved", "vs_map_packed", "vs_shard_bounds", "vs_resolve_hits", "vs_resolve_hits_mt",
    "vs_mapper_create", "vs_mapper_map", "vs_mapper_info", "vs_mapper_destroy", "vs_mapper_map_stream", "vs_map_records_stream",
    "vs_md_string", "vs_md_from_window", "vs_format_sam", "vs_bidir_index_main", "vs_bidir_mapping_main", "vs_vcf_loader_main", "vs_fasta_writer_main", "vs_bam_merger_main", "vs_bam_merger_ref_only_main", "vs_measure_int_peaks",
]

_lib = None


def lib():
    """Load the shared library (built by `make` / __graft_entry__.build())."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} is missing: run `make` (or __graft_entry__.build()); "
                          "varscot_b200 has no fallback implementation")
    L = C.CDLL(LIB_PATH)
    vp, u64, u32, i32 = C.c_void_p, C.c_uint64, C.c_uint32, C.c_int
    L.vs_packer_new.restype = vp
    L.vs_packer_free.argtypes = [vp]
    L.vs_packer_append.argtypes = [vp, C.c_char_p, C.c_size_t]
    L.vs_packer_end_contig.argtypes = [vp]
    L.vs_packer_finish.argtypes = [vp, C.POINTER(TextView)]
    L.vs_pack_text.argtypes = [vp, u64, vp, u32, vp, vp]
    L.vs_pack_text_planes.argtypes = [vp, u64, vp, u32, vp, vp, vp]
    L.vs_masks_from_planes.argtypes = [vp, vp, u64, vp]
    L.vs_masks_sparse.argtypes = [vp, u64, C.POINTER(vp), C.POINTER(u64)]
    L.vs_mask_source_build.argtypes = [vp, vp, u64, C.POINTER(MaskSource)]
    L.vs_mask_source_free.argtypes = [C.POINTER(MaskSource)]
    L.vs_text_save.argtypes = [C.c_char_p, C.POINTER(TextView)]
    L.vs_text_load.argtypes = [C.c_char_p, C.POINTER(TextView), C.POINTER(vp)]
    L.vs_text_masks.argtypes = [C.POINTER(TextView), vp]
    L.vs_map_records.argtypes = [C.POINTER(TextView), vp, u32, i32, i32, vp, i32, i32, C.POINTER(vp), C.POINTER(u64), C.POINTER(u64), C.POINTER(ScanStats)]
    L.vs_free.argtypes = [vp]
    L.vs_device_count.restype = i32
    L.vs_ctx_create.argtypes = [i32, C.POINTER(vp)]
    L.vs_ctx_destroy.argtypes = [vp]
    L.vs_last_error.restype = C.c_char_p; L.vs_last_error.argtypes = [vp]
    L.vs_ctx_set_chunk_words.argtypes = [vp, u64]
    L.vs_text_upload.argtypes = [vp, C.POINTER(TextView), u64, u64]
    L.vs_host_alloc.restype = vp; L.vs_host_alloc.argtypes = [C.c_size_t]
    L.vs_host_free.argtypes = [vp]
    L.vs_scan.argtypes = [vp, vp, u32, i32, i32, vp, u64, C.POINTER(u64), C.POINTER(ScanStats)]
    L.vs_scan_text.argtypes = [vp, C.POINTER(TextView), u64, u64, vp, u32, i32, i32, vp, u64, C.POINTER(u64), C.POINTER(ScanStats)]
    L.vs_scan_fetch.argtypes = [vp, vp, u64, C.POINTER(u64)]
    L.vs_scan_resolved.argtypes = [vp, C.POINTER(TextView), u64, u64, vp, u32, i32, i32, vp, u64, C.POINTER(u64), HIT_SINK, vp, C.POINTER(ScanStats)]
    L.vs_merge_resolved.argtypes = [vp, vp, i32, vp, C.POINTER(u64), i32]
    L.vs_ctx_set_option.argtypes = [vp, i32, C.c_int64]
    L.vs_index_drop.argtypes = [vp]
    L.vs_host_register.argtypes = [vp, C.c_size_t]
    L.vs_host_unregister.argtypes = [vp]
    L.vs_map_packed.argtypes = [C.POINTER(TextView), vp, u32, i32, i32, vp, i32, C.POINTER(vp), C.POINTER(u64), C.POINTER(ScanStats)]
    L.vs_shard_bounds.argtypes = [u64, i32, vp]
    L.vs_mapper_create.argtypes = [C.POINTER(TextView), vp, i32, C.POINTER(vp)]
    L.vs_mapper_map.argtypes = [vp, vp, u32, i32, i32, i32, C.POINTER(vp), C.POINTER(u64), C.POINTER(u64), C.POINTER(ScanStats)]
    L.vs_mapper_map_stream.argtypes = [vp, vp, u32, i32, i32, i32, u64, i32, RECORD_SINK, vp, C.POINTER(u64), C.POINTER(ScanStats)]
    L.vs_map_records_stream.argtypes = [C.POINTER(TextView), vp, u32, i32, i32, vp, i32, i32, u64, i32, RECORD_SINK, vp, C.POINTER(u64),
                                        C.POINTER(ScanStats)]
    L.vs_mapper_info.argtypes = [vp, C.POINTER(u32), C.POINTER(u64), C.POINTER(u64)]
    L.vs_mapper_destroy.argtypes = [vp]
    L.vs_resolve_hits.argtypes = [vp, u64, vp, u32, vp, C.POINTER(u64)]
    L.vs_resolve_hits_mt.argtypes = [vp, u64, vp, u32, vp, C.POINTER(u64), i32]
    L.vs_md_string.argtypes = [vp, u64, vp, i32, i32, C.c_char_p]
    L.vs_md_from_window.argtypes = [u64, vp, i32, i32, C.c_char_p]
    L.vs_format_sam.argtypes = [C.POINTER(Record), C.c_char_p, C.c_char_p, vp, C.c_char_p, C.c_char_p, C.c_size_t]
    L.vs_bidir_index_main.argtypes = [i32, C.POINTER(C.c_char_p)]
    L.vs_bidir_mapping_main.argtypes = [i32, C.POINTER(C.c_char_p)]
    L.vs_vcf_loader_main.argtypes = [i32, C.POINTER(C.c_char_p)]
    L.vs_fasta_writer_main.argtypes = [i32, C.POINTER(C.c_char_p)]
    L.vs_bam_merger_main.argtypes = [i32, C.POINTER(C.c_char_p)]
    L.vs_bam_merger_ref_only_main.argtypes = [i32, C.POINTER(C.c_char_p)]
    L.vs_measure_int_peaks.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    _lib = L
    return L


def check(rc: int, ctx=None):
    if rc != VS_OK:
        msg = lib().vs_last_error(ctx)
        raise VarscotError(rc, msg.decode() if msg else "")
