"""Resident mapper (vs_mapper_*, varscot_b200.Mapper): a text sharded once as vs_map_records shards it, every shard and its
candidate indexes kept in HBM across calls.

CPU: the device-memory estimate and the plan check of vs_mapper_create (tests/cpu_mapper_units.cpp), the refusal without a
device, argument errors.  GPU: Mapper.map against the oracle and against map_records on one device and on all devices; the
index lifecycle over repeated calls (extraction, bucketed build, bucketed scoring, re-extraction on a PAM change without a
new upload); argument errors that leave the resident state alone; two mappers on one device; the memory estimate against
what the contexts hold; a text beyond 4 Gbases held as two resident shards on one device."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

import varscot_b200 as V
from varscot_b200 import _lib
from tests.test_zz_beyond_4g import big, K as BIG_K  # noqa: F401  (module fixture: the ~4.55 Gbase text)
from tests.util import make_case

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PAT_BYTES_PER_GUIDE = 2 * 24 * 2              # pattern table: [2 strands][PAT_STRIDE = 24] uint16 per guide


def test_memory_estimate_and_plan_check_on_the_host(tmp_path):
    """vs::resident_shard_bytes grows with the shard's words, its PAM density, contigs and staged runs; vs::resident_plan_check
    accepts exactly the plans of 1-8 devices x 1-20 Gbases whose every device fits its free bytes (17 Gbases fit one 180 GB
    device as four shards, 30 Gbases do not)."""
    exe = str(tmp_path / "mapper_units")
    libdir = os.path.join(ROOT, "varscot_b200")
    r = subprocess.run(["g++", "-O1", "-std=c++20", "-pthread", "-fvisibility=hidden", "-o", exe,
                        os.path.join(ROOT, "tests", "cpu_mapper_units.cpp"), "-L" + libdir, "-lvarscot_scan", "-Wl,-rpath," + libdir],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "mapper units ok" in r.stdout, r.stdout + r.stderr


def test_mapper_create_without_a_device_fails_loudly():
    """In a child process that sees no device (so that the test runs on a GPU machine too): VS_ERR_NODEVICE with a message."""
    code = ("import sys; sys.path.insert(0, sys.argv[1])\n"
            "import pytest, varscot_b200 as V\n"
            "from varscot_b200 import _lib\n"
            "from tests.util import make_case\n"
            "c = make_case(seed=3, contig_lens=[5000, 45], n_guides=2, k=2)\n"
            "text = V.PackedText.from_ascii(c.ascii, c.offsets)\n"
            "with pytest.raises(V.VarscotError) as e:\n"
            "    V.Mapper(text)\n"
            "assert e.value.code == _lib.VS_ERR_NODEVICE and 'no CUDA device' in str(e.value), str(e.value)\n")
    r = subprocess.run([sys.executable, "-c", code, ROOT], capture_output=True, text=True, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert r.returncode == 0, r.stderr


def test_mapper_argument_errors():
    """NULL arguments and a view without contig offsets return VS_ERR_ARG before any device is touched."""
    L = _lib.lib()
    c = make_case(seed=3, contig_lens=[5000, 45], n_guides=2, k=2)
    text = V.PackedText.from_ascii(c.ascii, c.offsets)
    v = text.view()
    m = C.c_void_p()
    dev = np.zeros(1, dtype=np.int32)
    assert L.vs_mapper_create(None, dev.ctypes.data, 1, C.byref(m)) == _lib.VS_ERR_ARG and not m.value
    assert L.vs_mapper_create(C.byref(v), dev.ctypes.data, 1, None) == _lib.VS_ERR_ARG
    assert L.vs_mapper_create(C.byref(v), None, 1, C.byref(m)) == _lib.VS_ERR_ARG
    v.contig_off = None
    assert L.vs_mapper_create(C.byref(v), dev.ctypes.data, 1, C.byref(m)) == _lib.VS_ERR_ARG and not m.value
    assert b"contig offsets" in L.vs_last_error(None)
    rp, n = C.c_void_p(), C.c_uint64()
    g = np.zeros((1, 23), dtype=np.uint8)
    assert L.vs_mapper_map(None, g.ctypes.data, 1, 2, -1, 1, C.byref(rp), C.byref(n), None, None) == _lib.VS_ERR_ARG
    assert L.vs_mapper_info(None, None, None, None) == _lib.VS_ERR_ARG
    L.vs_mapper_destroy(None)


# ---- GPU ------------------------------------------------------------------------------------------------------------------
def _rows(rec):
    return list(zip(rec["guide"].tolist(), rec["flag"].tolist(), rec["contig"].tolist(), rec["pos"].tolist(), rec["mm"].tolist()))


@pytest.fixture(scope="module")
def planted():
    """Multi-contig text with empty, 22/23/45-base and long contigs, N runs, IUPAC codes and sites planted at contig starts and
    in last windows (tests/util.py)."""
    c = make_case(seed=41, contig_lens=[70000, 0, 45, 45, 23, 22, 31013, 1, 9000, 23, 50000], n_guides=8, k=8)
    return c, V.PackedText.from_ascii(c.ascii, c.offsets)


@pytest.fixture(scope="module")
def many_guides():
    """300 guides (above the bucketed-index threshold of 256) on a planted text of ~1 Mbases."""
    c = make_case(seed=43, contig_lens=[600000, 45, 23, 400000], n_guides=300, k=4, n_frac=0.001)
    return c, V.PackedText.from_ascii(c.ascii, c.offsets)


@pytest.mark.gpu
@pytest.mark.parametrize("all_devices", [False, True])
def test_mapper_equals_oracle_and_map_records(planted, all_devices):
    """Mapper.map at k = 0, 4, 6, 8, with and without -P, on one mapper (a PAM change re-extracts from the resident text):
    the oracle's records, order and flags included, and byte-identical to map_records on the same devices."""
    from oracle import oracle as O
    c, text = planted
    devices = list(range(V.device_count())) if all_devices else [0]
    if all_devices and len(devices) < 2:
        pytest.skip("one device visible")
    codes = O.text_codes(c.ascii)
    with V.Mapper(text, devices=devices) as m:
        for k in (0, 4, 6, 8):
            for pam in (None, "AG"):
                rec, coll, _ = m.map(c.guides, k, pam=pam, threads=4)
                want = [r[:5] for r in O.map_guides(codes, c.offsets, c.guides, k, pam=pam).rows()]
                assert _rows(rec) == want, (k, pam, len(rec), len(want))
                rec2, coll2, _ = V.map_records(text, c.guides, k, pam=pam, devices=devices, threads=4)
                assert rec.tobytes() == rec2.tobytes() and coll == coll2, (k, pam)
        assert len(want) > 0


@pytest.mark.gpu
def test_repeated_calls_reuse_the_resident_indexes(many_guides):
    """Call 1 extracts (index_reused 0), call 2 builds and scores the bucketed index (2, index_build_ms > 0), call 3 scores it
    (2, no build); all three return the records of map_records.  Alternating -P AG and no -P re-extracts each time from the
    resident text: the right records, and nothing travels to the device but the pattern table."""
    c, text = many_guides
    want = {pam: V.map_records(text, c.guides, c.k, pam=pam)[0] for pam in (None, "AG")}
    assert len(want[None]) > 0 and len(want["AG"]) >= len(want[None])
    with V.Mapper(text) as m:
        n_shards = m.n_shards
        runs = [m.map(c.guides, c.k) for _ in range(3)]
        assert [st.index_reused for _, _, st in runs] == [0, 2, 2]
        assert runs[1][2].index_build_ms > 0 and runs[2][2].index_build_ms == 0
        for rec, _, _ in runs:
            assert rec.tobytes() == want[None].tobytes()
        for pam in ("AG", None, "AG", None):
            rec, _, st = m.map(c.guides, c.k, pam=pam)
            assert rec.tobytes() == want[pam].tobytes(), pam
            assert st.index_reused == 0 and st.h2d_bytes == n_shards * len(c.guides) * PAT_BYTES_PER_GUIDE, (pam, st.h2d_bytes)


@pytest.mark.gpu
def test_argument_errors_leave_the_resident_indexes_alone(many_guides):
    """k = 9 and a guide code of 4 return VS_ERR_ARG; the next valid call still scores the bucketed index and returns the same
    records."""
    c, text = many_guides
    with V.Mapper(text) as m:
        m.map(c.guides, c.k)
        rec, _, st = m.map(c.guides, c.k)
        assert st.index_reused == 2
        bad = c.guides.copy()
        bad[5, 3] = 4
        for call in (lambda: m.map(c.guides, 9), lambda: m.map(bad, c.k)):
            with pytest.raises(V.VarscotError) as e:
                call()
            assert e.value.code == _lib.VS_ERR_ARG
        rec2, _, st2 = m.map(c.guides, c.k)
        assert st2.index_reused == 2 and st2.index_build_ms == 0 and rec2.tobytes() == rec.tobytes()


@pytest.mark.gpu
def test_two_mappers_on_one_device_genome_and_variant_segments():
    """A genome and the variant segments of a sample, each on its own mapper on device 0 at the same time (the resident genome
    plus a changing sample): each equals map_records of its own text, on the first call and on the resident second."""
    from varscot_b200 import synth, synth_core as core
    g = core.synth_genome(31, 3_000_000, 6, 0.05)
    genome = synth.from_planes(g)
    segments = synth.from_planes(core.synth_variant_segments(g, 32, 40_000))
    guides = core.synth_guides(33, 40)
    with V.Mapper(genome) as mg, V.Mapper(segments) as ms:
        for _ in range(2):
            for m, text in ((mg, genome), (ms, segments)):
                rec, _, _ = m.map(guides, 5, pam="AG", threads=4)
                want, _, _ = V.map_records(text, guides, 5, pam="AG", threads=4)
                assert len(want) > 0 and rec.tobytes() == want.tobytes()


@pytest.mark.gpu
def test_device_bytes_stay_within_the_create_time_estimate(many_guides):
    """After the bucketed build at 300 guides with -P AG (both candidate stores at the densest PAM set), the device memory the
    contexts hold is positive and at most the estimate vs_mapper_create checked against the free memory."""
    c, text = many_guides
    with V.Mapper(text) as m:
        assert 0 < m.device_bytes <= m.planned_bytes
        for _ in range(2):
            _, _, st = m.map(c.guides, c.k, pam="AG")
        assert st.index_reused == 2
        assert 0 < m.device_bytes <= m.planned_bytes, (m.device_bytes, m.planned_bytes)


@pytest.mark.gpu
def test_beyond_4g_text_stays_resident_as_two_shards_on_one_device(big):  # noqa: F811
    """The ~4.55 Gbase text of test_zz_beyond_4g: one device holds both shards resident; two maps return the records of
    map_records, the second from the resident indexes; with several devices visible, all devices give the same records."""
    text, guides, rec1, _, _ = big
    with V.Mapper(text, devices=[0]) as m:
        assert m.n_shards == 2
        for i in range(2):
            rec, _, st = m.map(guides, BIG_K, threads=8)
            assert rec.tobytes() == rec1.tobytes(), i
        assert st.index_reused >= 1
    n = V.device_count()
    if n > 1:
        with V.Mapper(text, devices=list(range(n))) as m:
            rec, _, _ = m.map(guides, BIG_K, threads=8)
            assert rec.tobytes() == rec1.tobytes()
