"""Streamed records (vs_mapper_map_stream, vs_map_records_stream, Mapper.map_stream, map_records_stream): the records of a map
delivered a range of whole guides at a time, optionally with each hit's 23-base genome window read on the device.

CPU: the streaming driver over fake shards (tests/cpu_stream_units.cpp); k_loc_windows against a naive gather and
vs_md_from_window against vs_md_string (tests/cpu_window_units.cpp); argument errors.  GPU: the concatenated deliveries against
Mapper.map / map_records byte for byte on the planted fixture, one device and all devices, several delivery sizes, and on the
~4.55 Gbase text held as two resident shards; windows against the text and MD:Z against md_string; the bytes windows add; an
abort that leaves the bucketed index resident; the bidir_mapping executable with many deliveries against one."""
import ctypes as C
import hashlib
import os
import subprocess

import numpy as np
import pytest

import varscot_b200 as V
from varscot_b200 import _lib
from tests.test_zz_beyond_4g import big, K as BIG_K  # noqa: F401  (module fixture: the ~4.55 Gbase text)
from tests.util import make_case, write_fasta, write_guides

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _build_and_run(tmp_path, name, ok):
    exe = str(tmp_path / name)
    libdir = os.path.join(ROOT, "varscot_b200")
    r = subprocess.run(["g++", "-O1", "-std=c++20", "-pthread", "-Wno-unknown-pragmas", "-fvisibility=hidden", "-o", exe,
                        os.path.join(ROOT, "tests", name + ".cpp"), "-L" + libdir, "-lvarscot_scan", "-Wl,-rpath," + libdir],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and ok in r.stdout, r.stdout + r.stderr[-4000:]


def test_stream_driver_over_fake_shards(tmp_path):
    """1-8 fake shards (empty ones, guides without hits), 0-300 guides, budgets of 1 record to unlimited: the deliveries
    concatenate to one vs_merge_resolved, collisions add up, ranges are contiguous whole guides within budget, windows follow
    their records, and a sink that aborts is not called again."""
    _build_and_run(tmp_path, "cpu_stream_units", "stream units ok")


def test_window_kernel_and_md_from_window_on_the_host(tmp_path):
    """k_loc_windows on shards with origin 0 and beyond 2^32 (first contig before the origin; first word, last word, halo) against
    a naive gather; vs_md_from_window equals vs_md_string at every window start, both styles and strands."""
    _build_and_run(tmp_path, "cpu_window_units", "window units ok")


def test_stream_argument_errors():
    """NULL sink, NULL text or mapper, and k = 9 return VS_ERR_ARG before any device is touched."""
    L = _lib.lib()
    c = make_case(seed=3, contig_lens=[5000, 45], n_guides=2, k=2)
    text = V.PackedText.from_ascii(c.ascii, c.offsets)
    v = text.view()
    g = np.ascontiguousarray(c.guides)
    dev = np.zeros(1, dtype=np.int32)
    null = C.cast(None, _lib.RECORD_SINK)
    sink = _lib.RECORD_SINK(lambda *a: 0)
    assert L.vs_map_records_stream(C.byref(v), g.ctypes.data, 2, 2, -1, dev.ctypes.data, 1, 1, 0, 0, null, None, None, None) == _lib.VS_ERR_ARG
    assert L.vs_map_records_stream(None, g.ctypes.data, 2, 2, -1, dev.ctypes.data, 1, 1, 0, 0, sink, None, None, None) == _lib.VS_ERR_ARG
    assert L.vs_map_records_stream(C.byref(v), g.ctypes.data, 2, 9, -1, dev.ctypes.data, 1, 1, 0, 0, sink, None, None, None) == _lib.VS_ERR_ARG
    assert L.vs_last_error(None).startswith(b"vs_map_records_stream: ")
    assert L.vs_mapper_map_stream(None, g.ctypes.data, 2, 2, -1, 1, 0, 0, sink, None, None, None) == _lib.VS_ERR_ARG
    assert V.md_from_window(0, np.zeros(23, np.uint8), 0) == "23"


# ---- GPU ------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def planted():
    c = make_case(seed=41, contig_lens=[70000, 0, 45, 45, 23, 22, 31013, 1, 9000, 23, 50000], n_guides=8, k=8)
    return c, V.PackedText.from_ascii(c.ascii, c.offsets)


@pytest.fixture(scope="module")
def many_guides():
    """300 guides (above the bucketed-index threshold of 256) on a planted text of ~1 Mbases."""
    c = make_case(seed=43, contig_lens=[600000, 45, 23, 400000], n_guides=300, k=4, n_frac=0.001)
    return c, V.PackedText.from_ascii(c.ascii, c.offsets)


class Collect:
    """A sink that keeps every delivery (copies: the views die with the call) and checks the contract as it goes."""

    def __init__(self, abort_at=None):
        self.rec, self.win, self.ranges, self.abort_at = [], [], [], abort_at

    def __call__(self, rec, win, lo, hi):
        assert not self.ranges or self.ranges[-1][1] == lo
        self.ranges.append((lo, hi, len(rec)))
        self.rec.append(rec.copy())
        if win is not None:
            self.win.append(win.copy())
        return self.abort_at is not None and len(self.ranges) - 1 == self.abort_at

    def records(self):
        return np.concatenate(self.rec) if self.rec else np.zeros(0, V.REC_DT)

    def windows(self):
        return np.concatenate(self.win) if self.win else np.zeros(0, np.uint64)


def _check_ranges(col, n_guides, budget):
    assert col.ranges[0][0] == 0 and col.ranges[-1][1] == n_guides
    for lo, hi, n in col.ranges:
        assert hi > lo and (n <= budget or hi - lo == 1), (lo, hi, n, budget)


def _decode(win):
    """windows -> (n, 23) Dna codes"""
    shifts = (2 * np.arange(23, dtype=np.uint64))
    return ((win[:, None] >> shifts[None, :]) & np.uint64(3)).astype(np.uint8)


def _text_codes(text, gpos):
    """(n, 23) Dna codes of the packed text at the given global window starts"""
    p = gpos[:, None].astype(np.int64) + np.arange(23)[None, :]
    w = text.bases[p >> 5]
    b = (p & 31).astype(np.uint32)
    return ((((w["hi"] >> b) & 1) << 1) | ((w["lo"] >> b) & 1)).astype(np.uint8)


@pytest.mark.gpu
@pytest.mark.parametrize("all_devices", [False, True])
def test_streamed_records_equal_the_one_shot_calls(planted, all_devices):
    """Mapper.map_stream and map_records_stream at k = 0, 4, 6, 8 with and without -P AG and records_per_delivery 0, 1 and about a
    third of the records: the concatenated deliveries are byte-identical to Mapper.map / map_records, collisions included."""
    c, text = planted
    devices = list(range(V.device_count())) if all_devices else [0]
    if all_devices and len(devices) < 2:
        pytest.skip("one device visible")
    with V.Mapper(text, devices=devices) as m:
        for k in (0, 4, 6, 8):
            for pam in (None, "AG"):
                want, coll, _ = m.map(c.guides, k, pam=pam, threads=4)
                want2, coll2, _ = V.map_records(text, c.guides, k, pam=pam, devices=devices, threads=4)
                assert want.tobytes() == want2.tobytes()
                for budget in (0, 1, max(1, len(want) // 3)):
                    col = Collect()
                    got_coll, st = m.map_stream(c.guides, k, col, pam=pam, threads=4, records_per_delivery=budget)
                    assert col.records().tobytes() == want.tobytes() and got_coll == coll, (k, pam, budget)
                    _check_ranges(col, len(c.guides), budget or (32 << 20))
                    assert st.n_hits == len(want)
                    col = Collect()
                    got_coll, _ = V.map_records_stream(text, c.guides, k, col, pam=pam, devices=devices, threads=4, records_per_delivery=budget)
                    assert col.records().tobytes() == want.tobytes() and got_coll == coll, (k, pam, budget)
                    _check_ranges(col, len(c.guides), budget or (32 << 20))
        assert len(want) > 0


@pytest.mark.gpu
def test_windows_are_the_text_and_give_md_string(planted):
    """Every window decodes to the text at offsets[contig] + pos; md_from_window equals md_string for every record (both styles);
    windows add exactly 8 B per hit to the device-to-host bytes."""
    c, text = planted
    with V.Mapper(text) as m:
        for k, pam in ((6, None), (8, "AG")):
            m.map(c.guides, k, pam=pam)                          # the index is resident: both streams below score it
            plain, with_win = Collect(), Collect()
            _, st0 = m.map_stream(c.guides, k, plain, pam=pam, records_per_delivery=50)
            _, st1 = m.map_stream(c.guides, k, with_win, pam=pam, records_per_delivery=50, windows=True)
            rec, win = with_win.records(), with_win.windows()
            assert rec.tobytes() == plain.records().tobytes() and len(win) == len(rec) > 0
            assert plain.win == []
            gpos = text.offsets[rec["contig"]].astype(np.int64) + rec["pos"].astype(np.int64)
            assert np.array_equal(_decode(win), _text_codes(text, gpos))
            for r, w, gp in zip(rec, win, gpos):
                g = c.guides[int(r["guide"])]
                strand = (int(r["flag"]) >> 4) & 1
                for style in (V.MD_SEQAN, V.MD_SAMTOOLS):
                    assert V.md_from_window(int(w), g, strand, style) == V.md_string(text, int(gp), g, strand, style)
            assert st1.d2h_bytes == st0.d2h_bytes + 8 * st1.n_hits, (st0.d2h_bytes, st1.d2h_bytes, st1.n_hits)


@pytest.mark.gpu
def test_abort_stops_the_stream_and_keeps_the_bucketed_index(many_guides):
    """Two maps build the bucketed index; a stream whose sink aborts on the second delivery raises VS_ERR_ARG ("the sink
    aborted") and is not called again; the next map returns the same records from the resident bucketed index, no rebuild."""
    c, text = many_guides
    with V.Mapper(text) as m:
        m.map(c.guides, c.k)
        want, _, st = m.map(c.guides, c.k)
        assert st.index_reused == 2 and len(want) > 10
        col = Collect(abort_at=1)
        with pytest.raises(V.VarscotError) as e:
            m.map_stream(c.guides, c.k, col, records_per_delivery=max(1, len(want) // 10))
        assert e.value.code == _lib.VS_ERR_ARG and "the sink aborted" in str(e.value)
        assert len(col.ranges) == 2
        rec, _, st = m.map(c.guides, c.k)
        assert rec.tobytes() == want.tobytes() and st.index_reused == 2 and st.index_build_ms == 0


@pytest.mark.gpu
def test_beyond_4g_two_resident_shards_stream(big):  # noqa: F811
    """The ~4.55 Gbase text as two resident shards on one device: at least 3 deliveries with windows concatenate to
    map_records' records, and every window is the text at the record's position."""
    text, guides, rec1, _, _ = big
    with V.Mapper(text, devices=[0]) as m:
        assert m.n_shards == 2
        col = Collect()
        budget = max(1, len(rec1) // 4)
        m.map_stream(guides, BIG_K, col, threads=8, records_per_delivery=budget, windows=True)
        assert len(col.ranges) >= 3
        assert col.records().tobytes() == rec1.tobytes()
        rec, win = col.records(), col.windows()
        gpos = text.offsets[rec["contig"]].astype(np.int64) + rec["pos"].astype(np.int64)
        assert np.array_equal(_decode(win), _text_codes(text, gpos))


@pytest.mark.gpu
def test_bidir_mapping_many_deliveries_write_the_same_sam(tmp_path, planted):
    """bidir_mapping with VARSCOT_RECORDS_PER_DELIVERY=1 (a delivery per guide) writes the SAM bytes of the default, at -T 1 and
    -T 8, with and without -P; on two devices too when visible."""
    c, _ = planted
    exe = os.path.join(ROOT, "build", "read_mapping_build", "bidir_mapping")
    genome, reads = str(tmp_path / "g.fa"), str(tmp_path / "r.fa")
    write_fasta(genome, c.names, c.ascii, c.offsets)
    write_guides(reads, range(len(c.guides)), c.guide_strs)
    gpu_sets = [None] + (["2"] if V.device_count() > 1 else [])
    for gpus in gpu_sets:
        for threads in (1, 8):
            for pam in (None, "AG"):
                digests = []
                for rpd in (None, "1"):
                    out = str(tmp_path / f"o_{threads}_{pam}_{rpd}_{gpus}.sam")
                    env = dict(os.environ)
                    env.pop("VARSCOT_RECORDS_PER_DELIVERY", None)
                    if rpd:
                        env["VARSCOT_RECORDS_PER_DELIVERY"] = rpd
                    if gpus:
                        env["VARSCOT_GPUS"] = gpus
                    args = [exe, "-G", genome, "-I", str(tmp_path / "idx"), "-R", reads, "-M", "6", "-T", str(threads), "-O", out]
                    if pam:
                        args += ["-P", pam]
                    r = subprocess.run(args, capture_output=True, text=True, env=env)
                    assert r.returncode == 0, r.stderr
                    data = open(out, "rb").read()
                    assert len(data) > 0
                    digests.append(hashlib.sha256(data).hexdigest())
                assert digests[0] == digests[1], (threads, pam, gpus)
