"""varscot_b200 — B200-native drop-in for VARSCOT's read_mapping stage (bidir_index / bidir_mapping).

Layout: csrc/ holds the hand-written sm_100a kernels and the C ABI (include/varscot_scan.h);
_lib.py binds it with ctypes; mapper.py mirrors the reference's two executables and exposes the
packed-text / scan-context objects; synth.py builds the synthetic workloads of BASELINE.json.
Importing the package loads libvarscot_scan.so and fails loudly if it is missing.
"""
from . import _lib
from ._lib import VarscotError, GLEN

_lib.lib()   # fail at import time, not at first use, when the CUDA library has not been built

from .mapper import (PackedText, ScanContext, Mapper, bidir_index, bidir_mapping, vcf_loader, fasta_writer, device_count, format_sam, guide_codes,  # noqa: E402
                     map_packed, map_records, map_records_stream, md_from_window, md_string, merge_resolved, pam_code, records_key_set, resolve_hits, shard_bounds, HIT_DT, LOC_DT, REC_DT, BASES_DT, MASKS_DT, SPARSE_DT,
                     MD_SEQAN, MD_SAMTOOLS)

__all__ = ["PackedText", "ScanContext", "Mapper", "bidir_index", "bidir_mapping", "vcf_loader", "fasta_writer", "device_count", "format_sam", "guide_codes",
           "map_packed", "map_records", "map_records_stream", "md_from_window", "md_string", "merge_resolved", "pam_code", "records_key_set", "resolve_hits", "shard_bounds", "VarscotError", "GLEN",
           "HIT_DT", "LOC_DT", "REC_DT", "BASES_DT", "MASKS_DT", "SPARSE_DT", "MD_SEQAN", "MD_SAMTOOLS"]
