"""Host-side mirror of the reference's read_mapping interface, on top of the C ABI.

The reference exposes this path only as two executables (VARSCOT_pipeline/read_mapping/bidir_index.cpp,
bidir_mapping.cpp); `bidir_index()` and `bidir_mapping()` below take the same options with the same meaning
and exit codes, and call the very same entry points the executables call.  The lower-level classes
(PackedText, ScanContext) are what bench.py and the parity tests drive.  All compute happens in the CUDA
library; nothing here scores windows.
"""
from __future__ import annotations

import ctypes as C
import numpy as np

from . import _lib
from ._lib import GLEN, Hit, Record, ScanStats, VarscotError, check

BASES_DT = np.dtype([("hi", "<u4"), ("lo", "<u4")])
MASKS_DT = np.dtype([("iv", "<u4"), ("lw", "<u4")])
SPARSE_DT = np.dtype([("word", "<u4"), ("iv", "<u4"), ("lw", "<u4")])
RUN_DT = np.dtype([("word", "<u4"), ("count", "<u4"), ("value", "<u4")])
HIT_DT = np.dtype([("pos", "<u4"), ("info", "<u4")])
LOC_DT = np.dtype([("key", "<u8"), ("contig", "<u4"), ("info", "<u4")])
REC_DT = np.dtype([("guide", "<u4"), ("contig", "<u4"), ("pos", "<u4"), ("flag", "<u2"), ("mm", "u1"), ("pad", "u1")])

MD_SEQAN, MD_SAMTOOLS = 0, 1

_GUIDE_LUT = np.zeros(256, dtype=np.uint8)
for _ch, _v in (("C", 1), ("G", 2), ("T", 3), ("U", 3)):
    _GUIDE_LUT[ord(_ch)] = _v
    _GUIDE_LUT[ord(_ch.lower())] = _v


def guide_codes(guides) -> np.ndarray:
    """23-nt guide strings -> (n, 23) Dna codes; non-ACGT -> A (bidir_mapping.cpp:194,256)."""
    out = np.zeros((len(guides), GLEN), dtype=np.uint8)
    for i, g in enumerate(guides):
        b = g.encode() if isinstance(g, str) else bytes(g)
        if len(b) != GLEN:
            raise ValueError(f"guide {i} is not {GLEN} nt")
        out[i] = _GUIDE_LUT[np.frombuffer(b, dtype=np.uint8)]
    return out


def pam_code(pam) -> int:
    """-P XY -> 4*x+y, or -1 when it can never match (bidir_mapping.cpp:240-247)."""
    if not pam:
        return -1
    lut = {"A": 0, "C": 1, "G": 2, "T": 3, "U": 3}
    if len(pam) != 2 or pam[0].upper() not in lut or pam[1].upper() not in lut:
        return -1
    return 4 * lut[pam[0].upper()] + lut[pam[1].upper()]


def _copy_array(ptr, count, dt):
    if not count:
        return np.zeros(0, dtype=dt)
    raw = np.ctypeslib.as_array(C.cast(ptr, C.POINTER(C.c_uint8)), shape=(count * dt.itemsize,))
    return raw.copy().view(dt)


class PackedText:
    """Bit-sliced text (include/varscot_scan.h): bases[n_words + 1] of {hi, lo}, window masks[n_words] of {iv, lw},
    the sparse form of the masks, contig offsets and optional names.  `view()` is the vs_text_view the C ABI takes."""

    def __init__(self, bases, masks, offsets, n_bases, names=None, sparse=None, source=None):
        self.bases = np.ascontiguousarray(bases, dtype=BASES_DT)
        self.masks = np.ascontiguousarray(masks, dtype=MASKS_DT)
        self.offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        self.n_bases = int(n_bases)
        self.names = names
        assert len(self.bases) == self.n_words + 1 and len(self.masks) == self.n_words
        if sparse is None:
            nz = np.flatnonzero((self.masks["iv"] | self.masks["lw"]) != 0)
            sparse = np.zeros(len(nz), dtype=SPARSE_DT)
            sparse["word"] = nz
            sparse["iv"] = self.masks["iv"][nz]
            sparse["lw"] = self.masks["lw"][nz]
        self.sparse = np.ascontiguousarray(sparse, dtype=SPARSE_DT)
        # compact mask source (include/varscot_scan.h): code bytes of the contig-end plane, its coded-block flags, N-plane runs,
        # end-plane runs
        self.em_code = self.em_dense = self.nm_runs = self.em_runs = None
        if source is not None:
            em_code, em_dense, nm_runs, em_runs = source
            self.em_code = np.ascontiguousarray(em_code, dtype=np.uint8)
            self.em_dense = np.ascontiguousarray(em_dense, dtype=np.uint8)
            self.nm_runs = np.ascontiguousarray(nm_runs, dtype=RUN_DT)
            self.em_runs = np.ascontiguousarray(em_runs, dtype=RUN_DT)
            assert len(self.em_code) == self.n_words + 1 and len(self.em_dense) == (self.n_words + 4096) // 4096
        self._pinned = []

    @property
    def n_words(self) -> int:
        return (self.n_bases + 31) // 32

    @property
    def n_contigs(self) -> int:
        return len(self.offsets) - 1

    @property
    def has_source(self) -> bool:
        return self.em_code is not None

    def view(self, use_sparse: bool = True, use_source: bool = True) -> _lib.TextView:
        """use_source: hand the compact mask source to the library when this text has one (uploads then move the planes and
        the device computes the masks); use_sparse: otherwise offer the sparse mask list."""
        v = _lib.TextView()
        v.n_bases, v.n_words, v.n_contigs, v.reserved = self.n_bases, self.n_words, self.n_contigs, 0
        v.contig_off = self.offsets.ctypes.data
        v.bases = self.bases.ctypes.data
        v.masks = self.masks.ctypes.data
        v.sparse = self.sparse.ctypes.data if use_sparse else None
        v.n_sparse = len(self.sparse) if use_sparse else 0
        if use_source and self.has_source:
            v.em_code, v.em_dense = self.em_code.ctypes.data, self.em_dense.ctypes.data
            v.nm_runs, v.em_runs = self.nm_runs.ctypes.data, self.em_runs.ctypes.data
            v.n_nm_runs, v.n_em_runs = len(self.nm_runs), len(self.em_runs)
        return v

    def _arrays(self):
        # what an upload reads: with a mask source the window masks never travel (the device computes them)
        return ("bases", "em_code", "em_dense", "nm_runs", "em_runs") if self.has_source else ("bases", "masks", "sparse")

    def pin(self):
        """Move bases, masks, sparse masks and the mask source into page-locked memory (vs_host_alloc) for full-speed H2D."""
        L = _lib.lib()
        for name in self._arrays():
            arr = getattr(self, name)
            nbytes = max(arr.nbytes, 16)
            p = L.vs_host_alloc(nbytes)
            if not p:
                raise VarscotError(_lib.VS_ERR_NOMEM, "vs_host_alloc failed")
            buf = (C.c_uint8 * nbytes).from_address(p)
            new = np.frombuffer(buf, dtype=arr.dtype, count=len(arr))
            new[:] = arr
            setattr(self, name, new)
            self._pinned.append(p)
        return self

    def unpin(self):
        L = _lib.lib()
        for name in self._arrays():
            setattr(self, name, np.array(getattr(self, name)))
        for p in self._pinned:
            L.vs_host_free(p)
        self._pinned = []

    @staticmethod
    def _with_source(bases, nm, em, offsets, n_bases, names) -> "PackedText":
        """Masks and the compact mask source from the N plane and the contig-end plane (n_words + 1 words each)."""
        L = _lib.lib()
        nw = (int(n_bases) + 31) // 32
        masks = np.zeros(nw, dtype=MASKS_DT)
        check(L.vs_masks_from_planes(nm.ctypes.data, em.ctypes.data, nw, masks.ctypes.data))
        ms = _lib.MaskSource()
        check(L.vs_mask_source_build(nm.ctypes.data, em.ctypes.data, nw, C.byref(ms)))
        try:
            source = (_copy_array(ms.em_code, nw + 1, np.dtype("u1")), _copy_array(ms.em_dense, int(ms.n_em_blocks), np.dtype("u1")),
                      _copy_array(ms.nm_runs, int(ms.n_nm_runs), RUN_DT), _copy_array(ms.em_runs, int(ms.n_em_runs), RUN_DT))
        finally:
            L.vs_mask_source_free(C.byref(ms))
        return PackedText(bases, masks, offsets, n_bases, names, source=source)

    @staticmethod
    def from_planes(hi, lo, nm, em, offsets, n_bases, names=None) -> "PackedText":
        """From bit planes of n_words + 1 words each (nm: N / padding plane, em: contig-end plane)."""
        nw = (int(n_bases) + 31) // 32
        nm = np.ascontiguousarray(nm, dtype=np.uint32)
        em = np.ascontiguousarray(em, dtype=np.uint32)
        bases = np.zeros(nw + 1, dtype=BASES_DT)
        bases["hi"][:nw] = np.asarray(hi[:nw], dtype=np.uint32) & ~nm[:nw]
        bases["lo"][:nw] = np.asarray(lo[:nw], dtype=np.uint32) & ~nm[:nw]
        return PackedText._with_source(bases, nm, em, offsets, n_bases, names)

    @staticmethod
    def from_ascii(ascii_bytes, offsets, names=None) -> "PackedText":
        L = _lib.lib()
        a = np.frombuffer(ascii_bytes, dtype=np.uint8) if isinstance(ascii_bytes, (bytes, bytearray)) else np.ascontiguousarray(ascii_bytes, dtype=np.uint8)
        off = np.ascontiguousarray(offsets, dtype=np.uint64)
        n = int(a.size)
        nw = (n + 31) // 32
        bases = np.zeros(nw + 1, dtype=BASES_DT)
        nm, em = np.zeros(nw + 1, dtype=np.uint32), np.zeros(nw + 1, dtype=np.uint32)
        check(L.vs_pack_text_planes(a.ctypes.data, n, off.ctypes.data, len(off) - 1, bases.ctypes.data, nm.ctypes.data, em.ctypes.data))
        return PackedText._with_source(bases, nm, em, off, n, names)

    @staticmethod
    def _from_view(v, names=None) -> "PackedText":
        nw = int(v.n_words)
        source = None
        if v.em_code and v.em_dense:
            source = (_copy_array(v.em_code, nw + 1, np.dtype("u1")), _copy_array(v.em_dense, (nw + 4096) // 4096, np.dtype("u1")),
                      _copy_array(v.nm_runs, int(v.n_nm_runs), RUN_DT), _copy_array(v.em_runs, int(v.n_em_runs), RUN_DT))
        if v.masks:
            masks = _copy_array(v.masks, nw, MASKS_DT)
        else:                                   # a cache written by bidir_index carries only the mask source
            masks = np.zeros(nw, dtype=MASKS_DT)
            check(_lib.lib().vs_text_masks(C.byref(v), masks.ctypes.data))
        return PackedText(_copy_array(v.bases, nw + 1, BASES_DT), masks,
                          _copy_array(v.contig_off, int(v.n_contigs) + 1, np.dtype("<u8")), int(v.n_bases), names,
                          _copy_array(v.sparse, int(v.n_sparse), SPARSE_DT) if v.sparse else None, source)

    @staticmethod
    def from_fasta(path: str) -> "PackedText":
        """Stream a FASTA through vs_packer_* exactly as bidir_index does."""
        L = _lib.lib()
        p = L.vs_packer_new()
        names = []
        try:
            have = False
            with open(path, "rb") as f:
                for line in f:
                    if line.startswith(b">"):
                        if have:
                            check(L.vs_packer_end_contig(p))
                        names.append(line[1:].rstrip(b"\r\n").decode())
                        have = True
                    elif have:
                        check(L.vs_packer_append(p, line, len(line)))
            if have:
                check(L.vs_packer_end_contig(p))
            v = _lib.TextView()
            check(L.vs_packer_finish(p, C.byref(v)))
            return PackedText._from_view(v, names)
        finally:
            L.vs_packer_free(p)

    def save(self, prefix: str):
        v = self.view()
        check(_lib.lib().vs_text_save(prefix.encode(), C.byref(v)))

    @staticmethod
    def load(prefix: str) -> "PackedText":
        L = _lib.lib()
        v, owner = _lib.TextView(), C.c_void_p()
        check(L.vs_text_load(prefix.encode(), C.byref(v), C.byref(owner)))
        try:
            return PackedText._from_view(v)
        finally:
            L.vs_free(owner)


class ScanContext:
    """One device context (vs_ctx): upload a shard of packed text, scan guides against it."""

    def __init__(self, device: int = 0):
        self._L = _lib.lib()
        self._ctx = C.c_void_p()
        check(self._L.vs_ctx_create(device, C.byref(self._ctx)))
        self.device = device
        self.last_stats = None

    def close(self):
        if self._ctx:
            self._L.vs_ctx_destroy(self._ctx)
            self._ctx = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_chunk_words(self, n: int):
        check(self._L.vs_ctx_set_chunk_words(self._ctx, n), self._ctx)

    def upload(self, text: PackedText, first_word: int = 0, n_words: int | None = None, use_sparse: bool = True, use_source: bool = True):
        """Make words [first_word, first_word + n_words) resident (vs_text_upload)."""
        if n_words is None:
            n_words = text.n_words - first_word
        v = text.view(use_sparse, use_source)
        check(self._L.vs_text_upload(self._ctx, C.byref(v), first_word, n_words), self._ctx)

    def _finish(self, rc, hits, n):
        if rc == _lib.VS_ERR_OVERFLOW:
            hits = np.zeros(n.value, dtype=HIT_DT)
            check(self._L.vs_scan_fetch(self._ctx, hits.ctypes.data, len(hits), C.byref(n)), self._ctx)
        else:
            check(rc, self._ctx)
        return hits[: n.value]

    def scan(self, guides: np.ndarray, k: int, pam=None, cap: int = 1 << 20, out: np.ndarray | None = None):
        """Scan the resident text (vs_scan). Returns (hits structured array, ScanStats). Hits are unordered, at global 32-bit
        positions: a resident shard of a text beyond 4 Gbases whose positions are shard-relative raises VarscotError
        (VS_ERR_ARG); scan_resolved serves it."""
        g = np.ascontiguousarray(guides, dtype=np.uint8).reshape(-1, GLEN)
        pc = pam if isinstance(pam, int) else pam_code(pam)
        hits = out if out is not None else np.zeros(cap, dtype=HIT_DT)
        n, st = C.c_uint64(), ScanStats()
        rc = self._L.vs_scan(self._ctx, g.ctypes.data, g.shape[0], k, pc, hits.ctypes.data, len(hits), C.byref(n), C.byref(st))
        hits = self._finish(rc, hits, n)
        self.last_stats = st
        return hits, st

    def scan_text(self, text: PackedText, guides: np.ndarray, k: int, pam=None, first_word: int = 0, n_words: int | None = None,
                  cap: int = 1 << 20, out: np.ndarray | None = None, use_sparse: bool = True, use_source: bool = True):
        """Upload (overlapped, chunk by chunk) and scan in one call (vs_scan_text): the end-to-end path.  Texts within 4 Gbases
        only (hits at global 32-bit positions); beyond, VarscotError (VS_ERR_ARG): use scan_resolved or map_records."""
        if n_words is None:
            n_words = text.n_words - first_word
        g = np.ascontiguousarray(guides, dtype=np.uint8).reshape(-1, GLEN)
        pc = pam if isinstance(pam, int) else pam_code(pam)
        hits = out if out is not None else np.zeros(cap, dtype=HIT_DT)
        n, st = C.c_uint64(), ScanStats()
        v = text.view(use_sparse, use_source)
        rc = self._L.vs_scan_text(self._ctx, C.byref(v), first_word, n_words, g.ctypes.data, g.shape[0], k, pc,
                                  hits.ctypes.data, len(hits), C.byref(n), C.byref(st))
        hits = self._finish(rc, hits, n)
        self.last_stats = st
        return hits, st

    def set_option(self, option: int, value: int):
        """vs_ctx_set_option: _lib.VS_OPT_KEEP_INDEX (keep the candidate index resident between scans), VS_OPT_HIT_CAPACITY."""
        check(self._L.vs_ctx_set_option(self._ctx, option, value), self._ctx)

    def drop_index(self):
        check(self._L.vs_index_drop(self._ctx), self._ctx)

    def scan_resolved(self, guides: np.ndarray, k: int, pam=None, text: PackedText | None = None, first_word: int = 0, n_words: int | None = None,
                      cap: int = 1 << 20, out: np.ndarray | None = None, sink=None):
        """vs_scan_resolved: hits resolved to (contig, pos) and sorted into emission order ON THE DEVICE.  text=None scans the
        resident shard, otherwise the shard is uploaded (overlapped) first.  sink(hits, guide_lo, guide_hi), if given, receives
        every guide super-chunk as a LOC_DT array (a view valid during the call only).  Returns (hits or None, ScanStats)."""
        g = np.ascontiguousarray(guides, dtype=np.uint8).reshape(-1, GLEN)
        pc = pam if isinstance(pam, int) else pam_code(pam)
        n, st = C.c_uint64(), ScanStats()
        v = text.view() if text is not None else None
        if text is not None and n_words is None:
            n_words = text.n_words - first_word
        vref = C.byref(v) if v is not None else None
        if sink is not None:
            def _cb(_user, ptr, cnt, lo, hi):
                arr = np.ctypeslib.as_array(C.cast(ptr, C.POINTER(C.c_uint8)), shape=(cnt * LOC_DT.itemsize,)).view(LOC_DT)
                return int(sink(arr, lo, hi) or 0)
            cb = _lib.HIT_SINK(_cb)
            rc = self._L.vs_scan_resolved(self._ctx, vref, first_word, n_words or 0, g.ctypes.data, g.shape[0], k, pc, None, 0, C.byref(n), cb, None, C.byref(st))
            check(rc, self._ctx)
            self.last_stats = st
            return None, st
        hits = out if out is not None else np.zeros(cap, dtype=LOC_DT)
        null_sink = C.cast(None, _lib.HIT_SINK)
        rc = self._L.vs_scan_resolved(self._ctx, vref, first_word, n_words or 0, g.ctypes.data, g.shape[0], k, pc, hits.ctypes.data, len(hits),
                                      C.byref(n), null_sink, None, C.byref(st))
        if rc == _lib.VS_ERR_OVERFLOW and out is None:
            # the caller's buffer was a guess: scan the (now resident) index again with room for every hit
            hits = np.zeros(n.value, dtype=LOC_DT)
            rc = self._L.vs_scan_resolved(self._ctx, None, 0, 0, g.ctypes.data, g.shape[0], k, pc, hits.ctypes.data, len(hits),
                                          C.byref(n), null_sink, None, C.byref(st))
        check(rc, self._ctx)
        self.last_stats = st
        return hits[: n.value], st

    def measure_int_peaks(self):
        a, b = C.c_double(), C.c_double()
        check(self._L.vs_measure_int_peaks(self._ctx, C.byref(a), C.byref(b)), self._ctx)
        return a.value, b.value


def device_count() -> int:
    n = _lib.lib().vs_device_count()
    return max(n, 0)


def map_packed(text: PackedText, guides: np.ndarray, k: int, pam=None, devices=None):
    """vs_map_packed: shard over devices, scan, return (hits, stats).  Texts within 4 Gbases only (hits at global 32-bit
    positions); beyond, VarscotError (VS_ERR_ARG): use map_records."""
    L = _lib.lib()
    g = np.ascontiguousarray(guides, dtype=np.uint8).reshape(-1, GLEN)
    dev = np.asarray(devices if devices else [0], dtype=np.int32)
    hp, n, st = C.c_void_p(), C.c_uint64(), ScanStats()
    v = text.view()
    check(L.vs_map_packed(C.byref(v), g.ctypes.data, g.shape[0], k, pam_code(pam) if not isinstance(pam, int) else pam,
                          dev.ctypes.data, len(dev), C.byref(hp), C.byref(n), C.byref(st)))
    try:
        hits = np.ctypeslib.as_array(C.cast(hp, C.POINTER(C.c_uint32)), shape=(n.value * 2,)).copy().view(HIT_DT) if n.value else np.zeros(0, HIT_DT)
    finally:
        L.vs_free(hp)
    return hits, st


def map_records(text: PackedText, guides: np.ndarray, k: int, pam=None, devices=None, threads: int = 1):
    """vs_map_records: what the bidir_mapping executable runs — shard over devices, scan with device-side hit resolution,
    merge.  Texts of any length: beyond 4 Gbases every device scans one or more shards of at most VS_MAX_SHARD_WORDS words
    one after the other.  Returns (records in emission order, key16_collisions, stats)."""
    L = _lib.lib()
    g = np.ascontiguousarray(guides, dtype=np.uint8).reshape(-1, GLEN)
    dev = np.asarray(devices if devices else [0], dtype=np.int32)
    rp, n, coll, st = C.c_void_p(), C.c_uint64(), C.c_uint64(), ScanStats()
    v = text.view()
    check(L.vs_map_records(C.byref(v), g.ctypes.data, g.shape[0], k, pam_code(pam) if not isinstance(pam, int) else pam,
                           dev.ctypes.data, len(dev), threads, C.byref(rp), C.byref(n), C.byref(coll), C.byref(st)))
    try:
        rec = _copy_array(rp, n.value, REC_DT) if n.value else np.zeros(0, REC_DT)
    finally:
        L.vs_free(rp)
    return rec, int(coll.value), st


def _record_sink(sink, windows: bool):
    """A RECORD_SINK that hands every delivery to sink(records REC_DT view, windows uint64 view or None, guide_lo, guide_hi) and
    aborts the stream when it returns a truthy value.  An exception in sink aborts the stream too and is kept in .error."""
    state = {"error": None}

    def _cb(_user, rp, wp, n, lo, hi):
        try:
            if n:
                rec = np.ctypeslib.as_array(C.cast(rp, C.POINTER(C.c_uint8)), shape=(n * REC_DT.itemsize,)).view(REC_DT)
                win = np.ctypeslib.as_array(C.cast(wp, C.POINTER(C.c_uint64)), shape=(n,)) if windows else None
            else:
                rec, win = np.zeros(0, REC_DT), (np.zeros(0, np.uint64) if windows else None)
            return 1 if sink(rec, win, lo, hi) else 0
        except BaseException as e:      # noqa: BLE001  (re-raised by the caller once the library has returned)
            state["error"] = e
            return 1

    return _lib.RECORD_SINK(_cb), state


def _finish_stream(rc, state, coll, st):
    if state["error"] is not None:
        raise state["error"]
    check(rc)
    return int(coll.value), st


def map_records_stream(text: PackedText, guides: np.ndarray, k: int, sink, pam=None, devices=None, threads: int = 1,
                       records_per_delivery: int = 0, windows: bool = False):
    """vs_map_records_stream: the records of map_records delivered a range of whole guides at a time, in emission order, while
    the devices score the next range.  sink(records, windows, guide_lo, guide_hi) receives REC_DT and (with windows=True) uint64
    views that are valid during the call only; a truthy return aborts (VarscotError VS_ERR_ARG).  records_per_delivery: target
    records per delivery (0 = 32 Mi).  Returns (key16_collisions, stats)."""
    L = _lib.lib()
    g = np.ascontiguousarray(guides, dtype=np.uint8).reshape(-1, GLEN)
    dev = np.asarray(devices if devices else [0], dtype=np.int32)
    coll, st = C.c_uint64(), ScanStats()
    cb, state = _record_sink(sink, windows)
    v = text.view()
    rc = L.vs_map_records_stream(C.byref(v), g.ctypes.data, g.shape[0], k, pam_code(pam) if not isinstance(pam, int) else pam,
                                 dev.ctypes.data, len(dev), threads, records_per_delivery, int(bool(windows)), cb, None,
                                 C.byref(coll), C.byref(st))
    return _finish_stream(rc, state, coll, st)


def md_from_window(window: int, guide: np.ndarray, strand: int, md_style: int = MD_SEQAN) -> str:
    """vs_md_from_window: the MD:Z value of a delivered record from its genome window (what md_string gives for it)."""
    buf = C.create_string_buffer(64)
    g = np.ascontiguousarray(guide, dtype=np.uint8)
    check(_lib.lib().vs_md_from_window(int(window), g.ctypes.data, strand, md_style, buf))
    return buf.value.decode()


class Mapper:
    """vs_mapper: map_records against a text kept resident in HBM.  The text is sharded over `devices` (default: device 0) as
    map_records shards it and uploaded once; every shard keeps its candidate indexes, so later calls with the same PAM set only
    score them (the bucketed index from the second call on, where the library's policy builds it).  Raises VarscotError with
    VS_ERR_NOMEM when the shards and their indexes would not fit the devices' free memory."""

    def __init__(self, text: PackedText, devices=None):
        self._L = _lib.lib()
        self._m = C.c_void_p()
        dev = np.asarray(devices if devices else [0], dtype=np.int32)
        v = text.view()
        check(self._L.vs_mapper_create(C.byref(v), dev.ctypes.data, len(dev), C.byref(self._m)))
        self.devices = [int(d) for d in dev]

    def map(self, guides: np.ndarray, k: int, pam=None, threads: int = 1):
        """Same as map_records(text, guides, k, pam, devices, threads): (records in emission order, key16_collisions, stats)."""
        g = np.ascontiguousarray(guides, dtype=np.uint8).reshape(-1, GLEN)
        rp, n, coll, st = C.c_void_p(), C.c_uint64(), C.c_uint64(), ScanStats()
        check(self._L.vs_mapper_map(self._m, g.ctypes.data, g.shape[0], k, pam_code(pam) if not isinstance(pam, int) else pam, threads,
                                    C.byref(rp), C.byref(n), C.byref(coll), C.byref(st)))
        try:
            rec = _copy_array(rp, n.value, REC_DT) if n.value else np.zeros(0, REC_DT)
        finally:
            self._L.vs_free(rp)
        return rec, int(coll.value), st

    def map_stream(self, guides: np.ndarray, k: int, sink, pam=None, threads: int = 1, records_per_delivery: int = 0,
                   windows: bool = False):
        """vs_mapper_map_stream: map()'s records delivered a range of whole guides at a time (see map_records_stream).  Returns
        (key16_collisions, stats)."""
        g = np.ascontiguousarray(guides, dtype=np.uint8).reshape(-1, GLEN)
        coll, st = C.c_uint64(), ScanStats()
        cb, state = _record_sink(sink, windows)
        rc = self._L.vs_mapper_map_stream(self._m, g.ctypes.data, g.shape[0], k, pam_code(pam) if not isinstance(pam, int) else pam,
                                          threads, records_per_delivery, int(bool(windows)), cb, None, C.byref(coll), C.byref(st))
        return _finish_stream(rc, state, coll, st)

    def _info(self):
        n, now, planned = C.c_uint32(), C.c_uint64(), C.c_uint64()
        check(self._L.vs_mapper_info(self._m, C.byref(n), C.byref(now), C.byref(planned)))
        return n.value, now.value, planned.value

    @property
    def n_shards(self) -> int:
        return self._info()[0]

    @property
    def device_bytes(self) -> int:
        """Device memory the mapper's contexts hold now."""
        return self._info()[1]

    @property
    def planned_bytes(self) -> int:
        """The create-time estimate of the device memory the resident shards need (all devices)."""
        return self._info()[2]

    def close(self):
        if self._m:
            self._L.vs_mapper_destroy(self._m)
            self._m = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def shard_bounds(n_words: int, n_shards: int) -> np.ndarray:
    """vs_shard_bounds: word ranges owned by each of n_shards ranks / devices."""
    out = np.zeros(n_shards + 1, dtype=np.uint64)
    check(_lib.lib().vs_shard_bounds(n_words, n_shards, out.ctypes.data))
    return out


def resolve_hits(hits: np.ndarray, offsets: np.ndarray, threads: int = 1):
    """vs_resolve_hits(_mt): reference emission order + flags. Returns (records, key16_collisions)."""
    L = _lib.lib()
    h = np.ascontiguousarray(hits, dtype=HIT_DT)
    off = np.ascontiguousarray(offsets, dtype=np.uint64)
    rec = np.zeros(len(h), dtype=REC_DT)
    coll = C.c_uint64()
    check(L.vs_resolve_hits_mt(h.ctypes.data, len(h), off.ctypes.data, len(off) - 1, rec.ctypes.data, C.byref(coll), threads))
    return rec, int(coll.value)


def merge_resolved(lists, threads: int = 1):
    """vs_merge_resolved: the device-sorted hit lists of the shards -> records in emission order with FLAGs.
    Returns (records, key16_collisions)."""
    L = _lib.lib()
    arrs = [np.ascontiguousarray(x, dtype=LOC_DT) for x in lists]
    ptrs = (C.c_void_p * max(1, len(arrs)))(*[a.ctypes.data for a in arrs])
    counts = np.array([len(a) for a in arrs] or [0], dtype=np.uint64)
    rec = np.zeros(int(sum(len(a) for a in arrs)), dtype=REC_DT)
    coll = C.c_uint64()
    check(L.vs_merge_resolved(ptrs, counts.ctypes.data, len(arrs), rec.ctypes.data, C.byref(coll), threads))
    return rec, int(coll.value)


def md_string(text: PackedText, gpos: int, guide: np.ndarray, strand: int, md_style: int = MD_SEQAN) -> str:
    buf = C.create_string_buffer(64)
    g = np.ascontiguousarray(guide, dtype=np.uint8)
    check(_lib.lib().vs_md_string(text.bases.ctypes.data, gpos, g.ctypes.data, strand, md_style, buf))
    return buf.value.decode()


def format_sam(rec, qname: str, rname: str, guide: np.ndarray, md: str) -> str:
    r = Record(int(rec["guide"]), int(rec["contig"]), int(rec["pos"]), int(rec["flag"]), int(rec["mm"]), 0)
    g = np.ascontiguousarray(guide, dtype=np.uint8)
    buf = C.create_string_buffer(len(qname) + len(rname) + 256)
    n = _lib.lib().vs_format_sam(C.byref(r), qname.encode(), rname.encode(), g.ctypes.data, md.encode(), buf, len(buf))
    if n < 0:
        raise VarscotError(_lib.VS_ERR_ARG, "vs_format_sam failed")
    return buf.raw[:n].decode()


def records_key_set(rec: np.ndarray):
    """Parity key (SURVEY.md 8a): (guide, strand bit, contig, pos, NM)."""
    return set(zip(rec["guide"].tolist(), ((rec["flag"] & 16) >> 4).tolist(), rec["contig"].tolist(), rec["pos"].tolist(), rec["mm"].tolist()))


def _main(fn, prog: str, args: list) -> int:
    argv = [prog.encode()] + [str(a).encode() for a in args]
    arr = (C.c_char_p * (len(argv) + 1))(*argv, None)
    return int(fn(len(argv), arr))


def bidir_index(genome: str, index: str) -> int:
    """`bidir_index -G genome -I index` (bidir_index.cpp:19-24). Returns the exit code."""
    return _main(_lib.lib().vs_bidir_index_main, "bidir_index", ["-G", genome, "-I", index])


def bidir_mapping(genome: str, index: str, reads: str, mismatches: int, output: str, threads: int = 1, pam: str | None = None,
                  md_style: str | None = None) -> int:
    """`bidir_mapping -G -I -R -M -T -O [-P]` (bidir_mapping.cpp:196-216). Returns the exit code."""
    args = ["-G", genome, "-I", index, "-R", reads, "-M", mismatches, "-T", threads, "-O", output]
    if pam:
        args += ["-P", pam]
    if md_style:
        args += ["--md-style", md_style]
    return _main(_lib.lib().vs_bidir_mapping_main, "bidir_mapping", args)


def vcf_loader(vcf: str, snp_fasta: str, genome: str, sample: int = 0, seq_length: int = 23, threads: int = 1) -> int:
    """`vcf_loader FILE.vcf SNPGENOME.fa GENOME.fa SAMPLE SEQLENGTH THREADS` (vcf_loader.cpp:13-17). Returns the exit code."""
    return _main(_lib.lib().vs_vcf_loader_main, "vcf_loader", [vcf, snp_fasta, genome, sample, seq_length, threads])


def fasta_writer(guides_fasta: str, flanking_fasta: str, bed: str, genome: str) -> int:
    """`fasta_writer OUTPUT1.fa OUTPUT2.fa ONTARGETS.bed GENOME.fa` (fasta_writer.cpp:11-15). Returns the exit code."""
    return _main(_lib.lib().vs_fasta_writer_main, "fasta_writer", [guides_fasta, flanking_fasta, bed, genome])
