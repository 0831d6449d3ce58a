"""Texts longer than 4 Gbases: shard-relative positions on the device and several shards per device.

CPU: the kernels that place positions (contig starts, hit resolution, extraction, bucket gather) run on the host with a
shard origin above 2^32 (tests/cpu_beyond_4g_units.cpp), the shard plan of vs_map_records, and the refusal of the
unordered calls.  GPU: a ~4.6 Gbase text (genome + a swarm of 45-base variant segments) with planted sites around 2^32, at
every shard border and in the last window of the text, against the oracle; one device against all devices; the
bidir_mapping executable on its packed-text cache; the unordered calls on a shard whose origin is not 0."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import varscot_b200 as V
from varscot_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MAX_SHARD_WORDS = (1 << 27) - 256              # VS_MAX_SHARD_WORDS (include/varscot_scan.h)


def test_beyond_4g_kernels_and_shard_plan_on_the_host(tmp_path):
    """k_contig_starts_* + k_resolve_hits on a shard whose origin lies above 2^32 (first contig starting before the origin,
    contigs ending on the shard border, empty contigs) against a 64-bit linear search; k_extract and k_bucket_gather with a
    non-zero position base against base 0; vs::shard_plan for 3.9 to 17 Gbases over 1, 2, 3 and 8 devices."""
    exe = str(tmp_path / "beyond_4g_units")
    libdir = os.path.join(ROOT, "varscot_b200")
    r = subprocess.run(["g++", "-O1", "-std=c++20", "-pthread", "-Wno-unknown-pragmas", "-fvisibility=hidden", "-o", exe,
                        os.path.join(ROOT, "tests", "cpu_beyond_4g_units.cpp"), "-L" + libdir, "-lvarscot_scan", "-Wl,-rpath," + libdir],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "beyond 4G units ok" in r.stdout, r.stdout + r.stderr


def _view_beyond_4g(n_bases):
    """A view that claims n_bases bases over tiny buffers: enough for calls that must refuse it before reading the text."""
    off = np.array([0, n_bases], dtype=np.uint64)
    bases = np.zeros(4, dtype=V.BASES_DT)
    v = _lib.TextView()
    v.n_bases, v.n_words, v.n_contigs = n_bases, (n_bases + 31) // 32, 1
    v.contig_off, v.bases, v.masks = off.ctypes.data, bases.ctypes.data, bases.ctypes.data
    return v, (off, bases)


def test_unordered_calls_refuse_texts_beyond_4g():
    """vs_map_packed and vs_scan_text report global 32-bit positions: on a view beyond 4 Gbases they fail with VS_ERR_ARG and
    point to the resolved calls, before any device is touched (vs_map_packed needs no context; vs_scan_text without one fails
    on the missing context first)."""
    L = _lib.lib()
    g = np.zeros((1, 23), dtype=np.uint8)
    v, keep = _view_beyond_4g((1 << 32) + 32 * 1000)
    hp, n = C.c_void_p(), C.c_uint64()
    dev = np.zeros(1, dtype=np.int32)
    rc = L.vs_map_packed(C.byref(v), g.ctypes.data, 1, 2, -1, dev.ctypes.data, 1, C.byref(hp), C.byref(n), None)
    assert rc == _lib.VS_ERR_ARG and not hp.value and n.value == 0
    assert b"vs_map_records" in L.vs_last_error(None)
    rc = L.vs_scan_text(None, C.byref(v), 0, v.n_words, g.ctypes.data, 1, 2, -1, None, 0, C.byref(n), None)
    assert rc == _lib.VS_ERR_ARG
    del keep


# ---- GPU ------------------------------------------------------------------------------------------------------------------
GENOME_BASES = 4_350_000_000                  # 2^32 falls inside the last chromosome of the ladder
N_VARIANTS = 2_500_000                        # ~200 Mbases of 45-base segments after the genome: ~4.55 Gbases in all
N_GUIDES, K = 24, 5
WINDOW = 256 << 20                            # bases of every oracle window


def _shard_borders(n_words):
    """Every shard border of the plans of 1 .. 8 devices (2, 3, 4, 6 and 8 shards at this size), in bases."""
    out = set()
    for s in (2, 3, 4, 6, 8):
        out.update(int(b) * 32 for b in V.shard_bounds(n_words, s)[1:-1])
    return sorted(out)


def _plant(p, gpos, w):
    """Write the 23 codes w over bases [gpos, gpos + 23) of the planes (N bits cleared)."""
    for i, c in enumerate(w.tolist()):
        q = gpos + i
        word, bit = q >> 5, np.uint32(1 << (q & 31))
        p.hi[word] = (p.hi[word] | bit) if c & 2 else (p.hi[word] & ~bit)
        p.lo[word] = (p.lo[word] | bit) if c & 1 else (p.lo[word] & ~bit)
        p.nm[word] &= ~bit


def _site_at(off, gpos):
    """The nearest window start at or after gpos whose 23 bases lie in one contig (or the last window before it)."""
    c = int(np.searchsorted(off, gpos, side="right")) - 1
    while int(off[c + 1]) - max(gpos, int(off[c])) < 23:
        c += 1
    return max(gpos, int(off[c]))


@pytest.fixture(scope="module")
def big():
    from varscot_b200 import synth, synth_core as core
    from tests.util import revcomp_codes
    rng = np.random.default_rng(77)
    g = core.synth_genome(21, GENOME_BASES, 24, 0.05)
    p = core.concat_texts(g, core.synth_variant_segments(g, 22, N_VARIANTS))
    guides = core.synth_guides(23, N_GUIDES)
    off = p.offsets.astype(np.int64)
    n_words = p.n_words
    assert n_words > MAX_SHARD_WORDS and int(off[24]) > (1 << 32)        # two shards on one device; 2^32 inside the genome
    # windows 23 bases apart around every border: the one at -1 straddles it, the one at -24 is the last before it
    want = [int(off[-1]) - 23]                               # the last window of the last contig (R4)
    for b in [1 << 32] + _shard_borders(n_words):
        want += [_site_at(off, b + d) for d in (-70, -47, -24, -1, 22)]
    sites = []
    for s in sorted(set(want)):
        if not sites or s >= sites[-1] + 23:                 # planted windows never overlap
            sites.append(s)
    for i, s in enumerate(sites):
        w = guides[i % N_GUIDES].copy()
        nm = int(rng.integers(0, K + 1)) if s != int(off[-1]) - 23 else 0
        if nm:
            idx = rng.choice(21, size=nm, replace=False)
            w[idx] = (w[idx] + rng.integers(1, 4, nm)) % 4
        _plant(p, s, revcomp_codes(w) if i % 2 else w)
    text = synth.from_planes(p)
    rec1, _, st1 = V.map_records(text, guides, K, devices=[0], threads=8)
    return text, guides, rec1, st1, sites


def _oracle_window_diff(rec, text, guides, s0, n):
    """Hit sets (guide, strand, global position, NM) of the scan and of the oracle run on bases [s0, s0 + n) alone; windows
    within 23 bases of a slice end that is not the text's end are left out (the slice cuts them)."""
    from oracle import oracle as O
    from varscot_b200 import synth
    s0 = s0 // 32 * 32
    n = min(n, text.n_bases - s0)
    real_end = s0 + n == text.n_bases
    hi = s0 + n - (0 if real_end else 23)
    gpos = text.offsets[rec["contig"]].astype(np.int64) + rec["pos"].astype(np.int64)
    sel = (gpos >= s0) & (gpos < hi)
    got = set(zip(rec["guide"][sel].tolist(), ((rec["flag"][sel] & 16) >> 4).tolist(), gpos[sel].tolist(), rec["mm"][sel].tolist()))
    off = synth.slice_offsets(text, s0, n)
    o = O.map_guides(synth.unpack_codes(text, s0, n), off, guides, K)
    opos = off[o.contig].astype(np.int64) + o.pos.astype(np.int64) + s0
    osel = opos < hi
    want = set(zip(o.guide[osel].tolist(), ((o.flag[osel] & 16) >> 4).tolist(), opos[osel].tolist(), o.mm[osel].tolist()))
    return got, want


@pytest.mark.gpu
def test_map_records_beyond_4g_equals_oracle_around_2p32_shard_borders_and_tail(big):
    """One device scans the ~4.55 Gbase text as two shards one after the other (the second with origin = its first base);
    the records equal the oracle's on windows of 256 Mbases around 2^32, around the shard border and at the tail, and every
    planted site is found."""
    text, guides, rec, st, sites = big
    n_words = text.n_words
    border = int(V.shard_bounds(n_words, 2)[1]) * 32
    assert n_words > MAX_SHARD_WORDS and st.n_hits == len(rec)
    gpos = text.offsets[rec["contig"]].astype(np.int64) + rec["pos"].astype(np.int64)
    found = set(gpos.tolist())
    assert all(s in found for s in sites), [s for s in sites if s not in found]
    for s0 in ((1 << 32) - WINDOW // 2, border - WINDOW // 2, text.n_bases - WINDOW):
        got, want = _oracle_window_diff(rec, text, guides, s0, WINDOW)
        assert len(want) > 10 and got == want, (s0, len(got), len(want), len(got ^ want))


@pytest.mark.gpu
def test_map_records_beyond_4g_one_device_equals_all_devices(big):
    """With several devices visible, the records of all devices (one or more shards each) are byte-identical to those of one
    device, flags included."""
    n = V.device_count()
    if n < 2:
        pytest.skip("one device visible")
    text, guides, rec1, _, _ = big
    rec, _, _ = V.map_records(text, guides, K, devices=list(range(n)), threads=8)
    assert rec.tobytes() == rec1.tobytes()


@pytest.mark.gpu
def test_bidir_mapping_on_a_packed_text_beyond_4g(big, tmp_path):
    """bidir_mapping -I on a .vsidx (+ .vsnames) written by PackedText.save for the text: exit 0, and its SAM rows are the
    records of map_records in the same order."""
    text, guides, rec, _, _ = big
    prefix = str(tmp_path / "big")
    text.save(prefix)
    with open(prefix + ".vsnames", "w") as f:
        f.write("".join(f"s{i}\n" for i in range(text.n_contigs)))
    genome = str(tmp_path / "unused.fa")
    open(genome, "w").close()                                # not read: the cache and its names are complete
    reads = str(tmp_path / "guides.fa")
    with open(reads, "w") as f:
        for i, g in enumerate(guides):
            f.write(f">g{i}\n" + "".join("ACGT"[c] for c in g) + "\n")
    sam = str(tmp_path / "out.sam")
    assert V.bidir_mapping(genome, prefix, reads, K, sam, threads=8) == 0
    rows = [ln.split("\t") for ln in open(sam).read().splitlines()]
    got = [(r[0], int(r[1]), r[2], int(r[3]) - 1, int(r[11].split(":")[2])) for r in rows]
    want = [(f"g{g}", f, f"s{c}", p, m) for g, f, c, p, m in zip(rec["guide"].tolist(), rec["flag"].tolist(), rec["contig"].tolist(),
                                                                  rec["pos"].tolist(), rec["mm"].tolist())]
    assert got == want and len(got) > 0


@pytest.mark.gpu
def test_unordered_scans_refuse_a_shard_beyond_4g_and_the_context_stays_usable(big):
    """vs_scan on a resident shard whose origin is not 0, and vs_scan_text on the text, return VS_ERR_ARG; vs_scan_resolved then
    scans the resident shard and finds the records of map_records that start in it."""
    text, guides, rec1, _, _ = big
    b = int(V.shard_bounds(text.n_words, 2)[1])
    with V.ScanContext(0) as ctx:
        ctx.upload(text, first_word=b)
        for call in (lambda: ctx.scan(guides, K), lambda: ctx.scan_text(text, guides, K, first_word=b)):
            with pytest.raises(_lib.VarscotError) as e:
                call()
            assert e.value.code == _lib.VS_ERR_ARG and "vs_scan_resolved" in str(e.value)
        hits, _ = ctx.scan_resolved(guides, K)
    rec, _ = V.merge_resolved([hits])
    gpos = text.offsets[rec1["contig"]].astype(np.int64) + rec1["pos"].astype(np.int64)
    assert len(rec) > 0 and V.records_key_set(rec) == V.records_key_set(rec1[gpos >= b * 32])
