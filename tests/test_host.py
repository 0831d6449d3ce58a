"""CPU tests of the product's host side: the C-ABI library loads and exports every declared symbol, the packer,
the packed-text cache, hit resolution (order + flags) and MD/SAM formatting agree with the oracle, the two
executables keep the reference's argv contract and exit codes, and nothing in the product reaches the oracle."""
import glob
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import varscot_b200 as V
from varscot_b200 import _lib
from oracle import oracle as O
from tests.util import GLEN, make_case, write_fasta, write_guides

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "build", "read_mapping_build")


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "varscot_scan.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = set(re.findall(r"\b(vs_[a-z0-9_]+)\s*\(", hdr))
    assert declared == set(_lib.EXPORTS), declared ^ set(_lib.EXPORTS)
    L = _lib.lib()
    for name in declared:
        assert getattr(L, name) is not None
    out = subprocess.run(["nm", "-D", "--defined-only", _lib.LIB_PATH], capture_output=True, text=True).stdout
    for name in declared:
        assert re.search(rf"\bT {name}\b", out), name


def test_library_contains_sm100a_kernels():
    out = subprocess.run(["cuobjdump", "-lelf", _lib.LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in out


def test_product_never_touches_the_oracle():
    srcs = glob.glob(os.path.join(ROOT, "varscot_b200", "**", "*.*"), recursive=True) + glob.glob(os.path.join(ROOT, "include", "*.h"))
    for f in srcs:
        if f.endswith((".so", ".pyc")):
            continue
        txt = open(f, errors="ignore").read()
        assert "vo_" not in txt and "libvo_oracle" not in txt and "from oracle" not in txt and "import oracle" not in txt, f


def test_no_device_fails_loudly():
    """In a child process that sees no device (so that the test runs on a GPU machine too)."""
    code = ("import sys; sys.path.insert(0, sys.argv[1])\n"
            "import pytest, varscot_b200 as V\n"
            "from varscot_b200 import _lib\n"
            "assert V.device_count() == 0\n"
            "with pytest.raises(V.VarscotError) as e:\n"
            "    V.ScanContext(0)\n"
            "assert e.value.code == _lib.VS_ERR_NODEVICE\n")
    r = subprocess.run([sys.executable, "-c", code, ROOT], capture_output=True, text=True, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert r.returncode == 0, r.stderr


def _expected_masks(codes, off):
    """Brute-force window masks (SURVEY.md R1, R3, R4) from Dna5 codes and contig offsets."""
    n = len(codes)
    nw = (n + 31) // 32
    iv = np.ones(nw * 32, np.uint8)
    lw = np.zeros(nw * 32, np.uint8)
    for c in range(len(off) - 1):
        s, e = int(off[c]), int(off[c + 1])
        for p in range(s, e - 22):
            if (codes[p:p + 23] < 4).all():
                iv[p] = 0
                lw[p] = 1 if p + 23 == e else 0
    return np.packbits(iv, bitorder="little").view("<u4"), np.packbits(lw, bitorder="little").view("<u4")


def test_pack_text_matches_numpy():
    rng = np.random.default_rng(0)
    lens = [100, 0, 37, 64, 5, 1, 31, 32, 33, 23, 22, 45]
    asc = bytes(rng.choice(np.frombuffer(b"ACGTACGTACGTACGTNacgtnRYuU*-", dtype=np.uint8), sum(lens)))
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    t = V.PackedText.from_ascii(asc, off)
    codes = O.text_codes(asc)
    n = len(codes)
    bits = lambda a: np.unpackbits(np.ascontiguousarray(a).view(np.uint8), bitorder="little")
    hi, lo = bits(t.bases["hi"]), bits(t.bases["lo"])
    assert ((hi[:n] * 2 + lo[:n])[codes < 4] == codes[codes < 4]).all()
    assert (hi[:n][codes == 4] == 0).all() and (lo[:n][codes == 4] == 0).all()
    assert (hi[n:] == 0).all() and (lo[n:] == 0).all()          # padding and the pad word are zero
    assert len(t.bases) == (n + 31) // 32 + 1 and len(t.masks) == (n + 31) // 32
    eiv, elw = _expected_masks(codes, off)
    assert (t.masks["iv"] == eiv).all() and (t.masks["lw"] == elw).all()
    nz = np.flatnonzero((t.masks["iv"] | t.masks["lw"]) != 0)
    assert t.sparse["word"].tolist() == nz.tolist() and (t.sparse["iv"] == t.masks["iv"][nz]).all() and (t.sparse["lw"] == t.masks["lw"][nz]).all()


def test_streaming_packer_and_fasta_quirks(tmp_path):
    case = make_case(3, [1000, 0, 45, 70, 71, 23], 1, 4)
    p = str(tmp_path / "g.fa")
    names = ["chr1 with description", "empty", "c_45", "c70", "c71", "c23"]
    write_fasta(p, names, case.ascii, case.offsets, width=70)
    a = V.PackedText.from_fasta(p)
    b = V.PackedText.from_ascii(case.ascii, case.offsets)
    assert a.n_bases == b.n_bases and a.offsets.tolist() == b.offsets.tolist() and a.names == names
    assert a.bases.tobytes() == b.bases.tobytes() and a.masks.tobytes() == b.masks.tobytes() and a.sparse.tobytes() == b.sparse.tobytes()
    # CRLF line ends, blank lines, no trailing newline, leading junk before the first header
    raw = open(p, "rb").read().replace(b"\n", b"\r\n")
    raw = b"junk line\r\n" + raw.rstrip(b"\r\n").replace(b">c70", b"\r\n>c70")
    p2 = str(tmp_path / "g2.fa")
    open(p2, "wb").write(raw)
    assert subprocess.run([os.path.join(BIN, "bidir_index"), "-G", p2, "-I", str(tmp_path / "i2")], capture_output=True).returncode == 0
    c = V.PackedText.load(str(tmp_path / "i2"))
    assert c.n_bases == b.n_bases and c.offsets.tolist() == b.offsets.tolist()
    assert c.bases.tobytes() == b.bases.tobytes() and c.masks.tobytes() == b.masks.tobytes() and c.sparse.tobytes() == b.sparse.tobytes()


def _expand_runs(runs, n):
    out = np.zeros(n, dtype=np.uint32)
    for w, c, v in zip(runs["word"].tolist(), runs["count"].tolist(), runs["value"].tolist()):
        assert v != 0 and c > 0 and (out[w:w + c] == 0).all()
        out[w:w + c] = v
    return out


def test_mask_source_reproduces_the_planes():
    """vs_mask_source_build: N-plane runs + contig-end plane (code bytes in coded blocks / runs elsewhere) expand to the planes they came from."""
    rng = np.random.default_rng(5)
    nw = 3 * 4096 + 100                       # four blocks of the contig-end plane, the last one partial
    nm = np.zeros(nw + 1, dtype=np.uint32)
    nm[10:5000] = 0xFFFFFFFF                  # one long run across a block border
    nm[5000] = 0x0000FFFF
    nm[9000:9003] = [1, 1, 2]                 # equal neighbours merge, a different value starts a new run
    nm[nw] = 0xFFFFFFFF
    em = np.zeros(nw + 1, dtype=np.uint32)
    em[17] = 1 << 5                           # block 0: sparse
    em[4096:8192] = np.uint32(1) << rng.integers(0, 32, 4096).astype(np.uint32)               # block 1: one end per word -> coded
    em[5000] = 0x80000001; em[5001] = 0x80000001; em[6000] = 0x00010100                       # ... except three words with two ends
    em[8192:8192 + 1300:1] = 7                # block 2: one run of 1300 equal words stays sparse
    em[12288 + 3] = 1 << 31                   # block 3 (partial): sparse
    t = V.PackedText.from_planes(np.zeros(nw + 1, np.uint32), np.zeros(nw + 1, np.uint32), nm, em, np.array([0, nw * 32], np.uint64), nw * 32)
    assert t.has_source and t.em_dense.tolist() == [0, 1, 0, 0]
    single = (em[4096:8192] & (em[4096:8192] - 1)) == 0
    code = t.em_code[4096:8192]
    assert (code[single] == np.log2(em[4096:8192][single]).astype(np.uint8)).all() and (code[~single] == 32).all()
    assert (t.em_code[:4096] == 32).all() and (t.em_code[8192:] == 32).all()
    assert _expand_runs(t.nm_runs, nw + 1).tolist() == nm.tolist()
    assert len(t.nm_runs) == 5 and t.nm_runs["count"].tolist() == [4990, 1, 2, 1, 1]
    sparse_part = em.copy(); sparse_part[4096:8192][single] = 0
    assert _expand_runs(t.em_runs, nw + 1).tolist() == sparse_part.tolist()
    assert len(t.em_runs) == 5                # word 17, run {5000, 2}, word 6000, the run of 1300, word 12291
    # the streaming packer builds the same source as the one-shot path
    lens = [700, 0, 45, 23, 5000]
    asc = bytes(rng.choice(np.frombuffer(b"ACGTN", dtype=np.uint8), sum(lens), p=[.24, .24, .24, .24, .04]))
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    a = V.PackedText.from_ascii(asc, off)
    assert a.has_source and len(a.em_code) == a.n_words + 1 and len(a.em_dense) == (a.n_words + 4096) // 4096


def _masks_from_source(t):
    """What the device does with a compact mask source (k_fill_runs, k_expand_em_code, k_masks_from_planes), in numpy."""
    import ctypes as C
    from varscot_b200 import _lib
    n = t.n_words + 1
    nm = _expand_runs(t.nm_runs, n)
    em = np.zeros(n, dtype=np.uint32)
    coded = np.repeat(t.em_dense.astype(bool), 4096)[:n]
    single = coded & (t.em_code < 32)
    em[single] = np.uint32(1) << t.em_code[single].astype(np.uint32)
    runs = _expand_runs(t.em_runs, n)
    em[runs != 0] = runs[runs != 0]
    masks = np.zeros(t.n_words, dtype=V.MASKS_DT)
    _lib.check(_lib.lib().vs_masks_from_planes(nm.ctypes.data, em.ctypes.data, t.n_words, masks.ctypes.data))
    return masks


@pytest.mark.parametrize("seed", range(6))
def test_mask_source_expands_to_the_packers_masks(seed):
    """Random texts (long contigs with N runs, swarms of 45-mers, contigs shorter than a window, empty contigs): the masks
    rebuilt from the compact source equal the masks the packer computed from the planes."""
    rng = np.random.default_rng(100 + seed)
    lens = []
    for _ in range(int(rng.integers(2, 6))):
        kind = rng.integers(0, 4)
        if kind == 0:
            lens += [int(rng.integers(50_000, 300_000))]
        elif kind == 1:
            lens += [45] * int(rng.integers(500, 6000))
        elif kind == 2:
            lens += rng.integers(0, 40, int(rng.integers(5, 400))).tolist()
        else:
            lens += rng.integers(30, 3000, int(rng.integers(5, 200))).tolist()
    total = int(sum(lens))
    asc = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, total)].copy()
    for _ in range(int(rng.integers(0, 4))):                       # N runs, some longer than a coded block
        a = int(rng.integers(0, max(1, total - 1)))
        asc[a:a + int(rng.integers(1, 200_000))] = ord("N")
    asc[rng.integers(0, total, total // 5000)] = ord("n")
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    t = V.PackedText.from_ascii(asc.tobytes(), off)
    got = _masks_from_source(t)
    assert got.tobytes() == t.masks.tobytes()


def test_text_cache_keeps_the_mask_source(tmp_path):
    case = make_case(9, [3000, 45, 45, 0, 23, 800], 1, 4)
    p = str(tmp_path / "g.fa")
    write_fasta(p, [f"c{i}" for i in range(6)], case.ascii, case.offsets, width=60)
    a = V.PackedText.from_fasta(p)
    b = V.PackedText.from_ascii(case.ascii, case.offsets)
    assert a.has_source and b.has_source
    for name in ("em_code", "em_dense", "nm_runs", "em_runs"):
        assert getattr(a, name).tobytes() == getattr(b, name).tobytes(), name
    a.save(str(tmp_path / "idx"))
    # with a source the window masks are not stored (the loader rebuilds them): bases + one code byte per word + small lists
    assert os.path.getsize(tmp_path / "idx.vsidx") < a.bases.nbytes + a.offsets.nbytes + a.em_code.nbytes + a.nm_runs.nbytes + a.em_runs.nbytes + 256
    u = V.PackedText.load(str(tmp_path / "idx"))
    assert u.has_source and u.masks.tobytes() == a.masks.tobytes() and u.sparse.tobytes() == a.sparse.tobytes()
    for name in ("em_code", "em_dense", "nm_runs", "em_runs"):
        assert getattr(u, name).tobytes() == getattr(a, name).tobytes(), name
    # a view without the source is saved without it, and loads without it
    v = a.view(use_source=False)
    import ctypes as C
    from varscot_b200 import _lib
    _lib.check(_lib.lib().vs_text_save(str(tmp_path / "plain").encode(), C.byref(v)))
    w = V.PackedText.load(str(tmp_path / "plain"))
    assert not w.has_source and w.masks.tobytes() == a.masks.tobytes() and w.bases.tobytes() == a.bases.tobytes()


def test_text_cache_roundtrip_and_errors(tmp_path):
    case = make_case(4, [500, 45, 45], 1, 4)
    t = V.PackedText.from_ascii(case.ascii, case.offsets)
    t.save(str(tmp_path / "idx"))
    u = V.PackedText.load(str(tmp_path / "idx"))
    assert u.n_bases == t.n_bases and u.offsets.tolist() == t.offsets.tolist() and u.bases.tobytes() == t.bases.tobytes()
    assert u.masks.tobytes() == t.masks.tobytes() and u.sparse.tobytes() == t.sparse.tobytes()
    with pytest.raises(V.VarscotError):
        V.PackedText.load(str(tmp_path / "missing"))
    open(str(tmp_path / "bad.vsidx"), "wb").write(b"not an index")
    with pytest.raises(V.VarscotError):
        V.PackedText.load(str(tmp_path / "bad"))


def _oracle_hits(case, k, pam=None):
    r = O.map_guides(O.text_codes(case.ascii), case.offsets, case.guides, k, pam=pam)
    hits = np.zeros(len(r), dtype=V.HIT_DT)
    hits["pos"] = (case.offsets[r.contig] + r.pos).astype(np.uint32)
    hits["info"] = (r.guide.astype(np.uint32) << 8) | (((r.flag & 16) >> 4).astype(np.uint32) << 7) | r.mm
    return r, hits


@pytest.mark.parametrize("seed,k", [(1, 4), (2, 6), (3, 8), (4, 0)])
def test_resolve_hits_reproduces_oracle_order_flags_md_sam(seed, k):
    """Feed the oracle's hits, shuffled, through the product's host pipeline: order, FLAG, MD and SAM must match."""
    case = make_case(seed, [40000, 45, 45, 0, 23, 9000], 6, k)
    r, hits = _oracle_hits(case, k)
    assert len(r) > 5
    rng = np.random.default_rng(seed)
    rec, coll = V.resolve_hits(hits[rng.permutation(len(hits))], case.offsets)
    assert coll == 0
    assert [(int(x["guide"]), int(x["flag"]), int(x["contig"]), int(x["pos"]), int(x["mm"])) for x in rec] == [x[:5] for x in r.rows()]
    text = V.PackedText.from_ascii(case.ascii, case.offsets)
    import ctypes as C
    for style in (V.MD_SEQAN, V.MD_SAMTOOLS):
        ro = O.map_guides(O.text_codes(case.ascii), case.offsets, case.guides, k, md_style=style)
        for i, x in enumerate(rec):
            md = V.md_string(text, int(case.offsets[x["contig"]]) + int(x["pos"]), case.guides[x["guide"]], (int(x["flag"]) >> 4) & 1, style)
            assert md == ro.md[i]
            if style == V.MD_SEQAN and i < 20:
                line = V.format_sam(x, f"g{x['guide']}", case.names[x["contig"]], case.guides[x["guide"]], md)
                buf = C.create_string_buffer(512)
                orec = O._Rec(int(ro.guide[i]), int(ro.contig[i]), int(ro.pos[i]), int(ro.flag[i]), int(ro.mm[i]), 0, ro.md[i].encode())
                n = O.lib().vo_format_sam(C.byref(orec), f"g{x['guide']}".encode(), case.names[x["contig"]].encode(),
                                          case.guides[x["guide"]].ctypes.data, buf, 512)
                assert line == buf.raw[:n].decode()
                assert len(line.rstrip("\n").split("\t")) == 13


def test_resolve_hits_wide_key_order_and_collision_count():
    nct = 65536 + 3
    off = (np.arange(nct + 1) * 45).astype(np.uint64)
    hits = np.zeros(4, dtype=V.HIT_DT)
    # same guide/strand: contigs 2, 65538 (same id16, same pos), 1, 65537 (same id16, different pos)
    hits["pos"] = [2 * 45 + 5, 65538 * 45 + 5, 1 * 45 + 7, 65537 * 45 + 3]
    hits["info"] = [(0 << 8) | 2, (0 << 8) | 1, (0 << 8) | 3, (0 << 8) | 3]
    rec, coll = V.resolve_hits(hits, off)
    assert coll == 1
    # key order: (id16=1,pos=3,c=65537) (1,7,c=1) (2,5,c=2) (2,5,c=65538); running best -> emission
    key = [(65537, 3), (1, 3), (2, 2), (65538, 1)]
    exp = []
    best = 0
    for i in range(1, 4):
        if key[i][1] >= key[best][1]:
            exp.append((key[i][0], 256))
        else:
            exp.append((key[best][0], 256)); best = i
    exp.append((key[best][0], 0))
    assert [(int(x["contig"]), int(x["flag"])) for x in rec] == exp


def test_golden_rows_roundtrip_through_host_pipeline():
    for path in sorted(glob.glob(os.path.join(ROOT, "tests", "golden", "case_*.json"))):
        d = json.load(open(path))
        off = np.array(d["offsets"], dtype=np.uint64)
        hits = np.zeros(len(d["rows"]), dtype=V.HIT_DT)
        for i, (g, flag, c, pos, mm, md) in enumerate(d["rows"]):
            hits[i] = (int(off[c]) + pos, (g << 8) | (((flag >> 4) & 1) << 7) | mm)
        rec, _ = V.resolve_hits(hits[::-1].copy(), off)
        text = V.PackedText.from_ascii(d["ascii"].encode(), off)
        guides = V.guide_codes(d["guides"])
        got = [[int(x["guide"]), int(x["flag"]), int(x["contig"]), int(x["pos"]), int(x["mm"]),
                V.md_string(text, int(off[x["contig"]]) + int(x["pos"]), guides[x["guide"]], (int(x["flag"]) >> 4) & 1)] for x in rec]
        assert got == d["rows"]


def test_shard_bounds_cover_text_once():
    for nw, n in ((0, 1), (1, 1), (255, 2), (256, 2), (1000, 3), (100000, 8), (110987654, 8)):
        b = V.shard_bounds(nw, n)
        assert b[0] == 0 and b[-1] == nw and (np.diff(b.astype(np.int64)) >= 0).all()
        assert all(int(x) % 256 == 0 for x in b[1:-1])
        if nw > 256 * n * 8:
            sizes = np.diff(b.astype(np.int64))
            assert sizes.max() - sizes.min() <= 512


def run_cli(prog, *args):
    return subprocess.run([os.path.join(BIN, prog), *map(str, args)], capture_output=True, text=True)


def test_cli_contract_exit_codes(tmp_path):
    case = make_case(9, [2000], 2, 4)
    g, r = str(tmp_path / "g.fa"), str(tmp_path / "r.fa")
    write_fasta(g, ["chr1"], case.ascii, case.offsets)
    write_guides(r, ["a", "b"], case.guide_strs)
    # bidir_index: stdout lines of bidir_index.cpp:42,49
    x = run_cli("bidir_index", "-G", g, "-I", tmp_path / "idx")
    assert x.returncode == 0 and x.stdout == "Number of sequences: 1\nIndex created successfully\n"
    assert os.path.exists(tmp_path / "idx.vsidx")
    assert run_cli("bidir_index", "--genome", g, "--index", tmp_path / "idx2").returncode == 0
    assert run_cli("bidir_index", "-G", g).returncode == 1                                  # missing required -I
    assert run_cli("bidir_index", "-G", tmp_path / "g.txt", "-I", tmp_path / "i").returncode == 1   # extension validation
    assert run_cli("bidir_index", "-G", tmp_path / "nope.fa", "-I", tmp_path / "i").returncode == 1
    assert run_cli("bidir_index", "-h").returncode == 0
    # bidir_mapping: parse errors -> 1 (bidir_mapping.cpp:219-220), k outside 0..8 -> 1 with the reference's message (:234-238)
    base = ["-G", g, "-I", tmp_path / "idx", "-R", r, "-O", tmp_path / "o.sam"]
    x = run_cli("bidir_mapping", *base, "-M", 9)
    assert x.returncode == 1 and "Maximum number of mismatches must lie between 0 and 8" in x.stderr
    assert run_cli("bidir_mapping", *base, "-M", -1).returncode == 1
    assert run_cli("bidir_mapping", *base).returncode == 1                                   # -M required
    assert run_cli("bidir_mapping", *base, "-M", "x").returncode == 1
    assert run_cli("bidir_mapping", "-G", g, "-I", tmp_path / "idx", "-R", r, "-M", 4, "-O", tmp_path / "o.txt").returncode == 1
    assert run_cli("bidir_mapping", *base, "-M", 4, "--bogus").returncode == 1
    assert run_cli("bidir_mapping", "--help").returncode == 0
    x = run_cli("bidir_mapping", "-G", g, "-I", tmp_path / "idx", "-R", r, "-M", 4, "-O", tmp_path / "nodir" / "o.sam")
    assert x.returncode == 1 and "Could not open output path" in x.stderr
    # wrong guide length is refused
    write_guides(str(tmp_path / "bad.fa"), ["a"], ["ACGT"])
    assert run_cli("bidir_mapping", "-G", g, "-I", tmp_path / "idx", "-R", tmp_path / "bad.fa", "-M", 4, "-O", tmp_path / "o.sam").returncode == 1
    x = subprocess.run([os.path.join(BIN, "bidir_mapping"), *map(str, base), "-M", "4"], capture_output=True, text=True,
                       env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))              # no device visible, on a GPU machine too
    assert x.returncode == 1 and "no usable CUDA device" in x.stderr and "Reads loaded (total: 2)." in x.stdout


def test_resolve_hits_threads_agree():
    """vs_resolve_hits_mt with 1, 3 and 8 threads produces the same records (and the same collision count)."""
    rng = np.random.default_rng(12)
    nct = 70000
    off = (np.arange(nct + 1) * 45).astype(np.uint64)
    n = 60000
    hits = np.zeros(n, dtype=V.HIT_DT)
    hits["pos"] = rng.integers(0, nct, n) * 45 + rng.integers(0, 23, n)
    hits["info"] = (rng.integers(0, 37, n).astype(np.uint32) << 8) | (rng.integers(0, 2, n).astype(np.uint32) << 7) | rng.integers(0, 7, n).astype(np.uint32)
    hits = np.unique(hits)                      # a scan never reports the same (pos, guide, strand) twice
    ref, c1 = V.resolve_hits(hits, off, threads=1)
    for t in (3, 8):
        got, c = V.resolve_hits(hits[rng.permutation(len(hits))], off, threads=t)
        assert got.tobytes() == ref.tobytes() and c == c1
    assert c1 > 0 and len(ref) == len(hits)


def test_device_code_on_the_host(tmp_path):
    """vs_kernels.cuh compiled for the host (tests/cpu_kernel_units.cpp): k_score<K> for every k and the mask kernels run thread
    by thread from their real source against naive restatements; k_extract's phase 2 runs through the very text the kernel
    includes (vs_extract_block.inc, plus the experimental half-block variant); transposes, candidate masks, adders, <= k tests,
    pattern table and plane layout have their own checks.  Launch geometry, streams and ptxas are what the gpu tests add."""
    exe = str(tmp_path / "kernel_units")
    src = os.path.join(ROOT, "tests", "cpu_kernel_units.cpp")
    r = subprocess.run(["g++", "-O1", "-std=c++20", "-pthread", "-Wno-unknown-pragmas", "-o", exe, src], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 0 and "kernel helper units ok" in r.stdout, r.stdout + r.stderr


def _loc_lists_from_hits(hits, offsets, n_lists, rng):
    """What vs_scan_resolved delivers, built on the host: hits -> (key, contig, info), dealt to n_lists shards, each sorted."""
    off = np.asarray(offsets, dtype=np.uint64)
    starts = off[:-1]
    # last contig whose start is <= pos (empty contigs share a start; the non-empty one is the last)
    contig = np.searchsorted(starts, hits["pos"].astype(np.uint64), side="right") - 1
    pos = hits["pos"].astype(np.uint64) - starts[contig]
    info = hits["info"].astype(np.uint64)
    loc = np.zeros(len(hits), dtype=V.LOC_DT)
    loc["key"] = ((info >> np.uint64(8)) << np.uint64(49)) | (((info >> np.uint64(7)) & np.uint64(1)) << np.uint64(48)) | \
                 ((contig.astype(np.uint64) & np.uint64(0xFFFF)) << np.uint64(32)) | pos
    loc["contig"] = contig
    loc["info"] = hits["info"]
    owner = rng.integers(0, n_lists, len(hits))
    out = []
    for l in range(n_lists):
        part = loc[owner == l]
        out.append(part[np.argsort(part["key"], kind="stable")])
    return out


@pytest.mark.parametrize("n_lists,threads", [(1, 1), (1, 4), (3, 1), (8, 5)])
def test_merge_resolved_equals_resolve_hits(n_lists, threads):
    """vs_merge_resolved over device-style sorted shard lists == vs_resolve_hits over the raw hits: same records, same order,
    same FLAGs, same collision count — incl. > 65536 contigs (ties on the 16-bit key are ordered by the full id)."""
    rng = np.random.default_rng(100 + n_lists)
    nct = 70000
    off = np.concatenate([[0], np.cumsum(rng.integers(0, 60, nct))]).astype(np.uint64)       # incl. empty contigs
    n = 30000
    hits = np.zeros(n, dtype=V.HIT_DT)
    hits["pos"] = rng.integers(0, int(off[-1]), n)
    # provoke 16-bit key collisions: copies of some hits moved by whole multiples of 65536 contigs are unlikely at random, so
    # build them: same guide / strand / in-contig position in contig c and c + 65536
    lens = np.diff(off.astype(np.int64))
    for c in range(0, 4000, 7):
        if lens[c] > 5 and lens[c + 65536] > 5:
            hits["pos"][c] = off[c] + 3
            hits["pos"][c + 1] = off[c + 65536] + 3
    guide = rng.integers(0, 40, n).astype(np.uint32)
    strand = rng.integers(0, 2, n).astype(np.uint32)
    guide[1:4000:7] = guide[0:3999:7]; strand[1:4000:7] = strand[0:3999:7]
    hits["info"] = (guide << 8) | (strand << 7) | rng.integers(0, 7, n).astype(np.uint32)
    hits = np.unique(hits)                                    # a scan never reports a (pos, guide, strand) twice
    _, first = np.unique(np.stack([hits["pos"], hits["info"] >> 7], axis=1), axis=0, return_index=True)
    hits = hits[np.sort(first)]
    want, coll_want = V.resolve_hits(hits, off)
    lists = _loc_lists_from_hits(hits, off, n_lists, rng)
    got, coll = V.merge_resolved(lists, threads=threads)
    assert got.tolist() == want.tolist()
    assert coll == coll_want and coll > 0


def test_merge_resolved_empty_lists():
    rec, coll = V.merge_resolved([np.zeros(0, V.LOC_DT), np.zeros(0, V.LOC_DT)])
    assert len(rec) == 0 and coll == 0
    rec, coll = V.merge_resolved([])
    assert len(rec) == 0
