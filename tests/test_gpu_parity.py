"""GPU parity tests: the CUDA path, called through the C ABI, against the CPU oracle on the same seeded
inputs.  Bit-exact: record lists (guide, FLAG, contig, pos, NM) must be identical, in the same order."""
import os
import subprocess

import numpy as np
import pytest

from tests.util import GLEN, make_case, revcomp_codes, write_fasta, write_guides

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "build", "read_mapping_build")


def oracle_rows(ascii_bytes, offsets, guides, k, pam=None):
    from oracle import oracle as O
    r = O.map_guides(O.text_codes(ascii_bytes), offsets, guides, k, pam=pam)
    return r.rows()


def gpu_rows(ascii_bytes, offsets, guides, k, pam=None, shards=1, with_md=True, chunk_words=None, streamed=False, use_sparse=True, use_source=True):
    import varscot_b200 as V
    text = V.PackedText.from_ascii(ascii_bytes, offsets)
    parts = []
    nw = text.n_words
    bounds = [nw * i // shards for i in range(shards + 1)]
    for i in range(shards):
        if bounds[i + 1] <= bounds[i]:
            continue
        with V.ScanContext(0) as ctx:
            if chunk_words:
                ctx.set_chunk_words(chunk_words)
            if streamed:
                hits, _ = ctx.scan_text(text, guides, k, pam=pam, first_word=bounds[i], n_words=bounds[i + 1] - bounds[i], cap=1 << 12,
                                        use_sparse=use_sparse, use_source=use_source)
            else:
                ctx.upload(text, bounds[i], bounds[i + 1] - bounds[i], use_sparse=use_sparse, use_source=use_source)
                hits, _ = ctx.scan(guides, k, pam=pam, cap=1 << 12)
            parts.append(hits.copy())
    hits = np.concatenate(parts) if parts else np.zeros(0, V.HIT_DT)
    rec, _ = V.resolve_hits(hits, offsets)
    rows = []
    for r in rec:
        md = V.md_string(text, int(offsets[r["contig"]]) + int(r["pos"]), guides[r["guide"]], (int(r["flag"]) >> 4) & 1) if with_md else ""
        rows.append((int(r["guide"]), int(r["flag"]), int(r["contig"]), int(r["pos"]), int(r["mm"]), md))
    return rows


def assert_same(case, shards=1, **kw):
    exp = oracle_rows(case.ascii, case.offsets, case.guides, case.k, case.pam)
    got = gpu_rows(case.ascii, case.offsets, case.guides, case.k, case.pam, shards=shards, **kw)
    assert len(got) == len(exp), f"{len(got)} GPU records vs {len(exp)} oracle records"
    assert got == exp
    return len(exp)


@pytest.mark.parametrize("k", list(range(9)))
def test_all_k(k):
    case = make_case(seed=100 + k, contig_lens=[20000, 45, 3000, 0, 23, 46, 10000], n_guides=5, k=k)
    n = assert_same(case)
    assert n > 0


@pytest.mark.parametrize("pam", [None, "AG", "TT", "CC", "GG"])
def test_extra_pam(pam):
    case = make_case(seed=7, contig_lens=[30000, 5000], n_guides=4, k=4, pam=pam, guide_pam=(pam or "GG"))
    assert_same(case)


def test_many_guides_chunking():
    # > 512 guides exercises several constant-memory pattern chunks per strand
    case = make_case(seed=11, contig_lens=[40000], n_guides=1100, k=3, plant=False)
    rng = np.random.default_rng(5)
    codes = np.frombuffer(case.ascii, dtype=np.uint8).copy()
    lut = np.frombuffer(b"ACGT", dtype=np.uint8)
    for g in (0, 511, 512, 513, 1023, 1024, 1099):
        p = int(rng.integers(0, 40000 - GLEN))
        w = case.guides[g].copy()
        if g % 2:
            w = revcomp_codes(w)
        codes[p:p + GLEN] = lut[w]
    case.ascii = bytes(codes)
    n = assert_same(case)
    assert n >= 7


def test_edge_contigs():
    """L < 23, L == 23, last-window rule R4 both ways, first window, N at every offset."""
    rng = np.random.default_rng(3)
    g = rng.integers(0, 4, GLEN).astype(np.uint8); g[21:] = 2
    lut = np.frombuffer(b"ACGT", dtype=np.uint8)
    contigs = []
    k = 4
    # exact-length contigs: perfect, H2 <= K and H2 > K variants (K = 2)
    for mm_pos in ([], [0, 1, 2], [12, 13], [12, 13, 14], [0, 12, 13, 14], [11, 15, 20], [3, 4, 5, 6]):
        for strand in (0, 1):
            w = g.copy()
            for p in mm_pos:
                w[p] = (w[p] + 1) % 4
            w[21:] = 2
            if strand:
                w = revcomp_codes(w)
            contigs.append(lut[w])
            contigs.append(np.concatenate([lut[rng.integers(0, 4, 22)], lut[w]]))          # site is the LAST window of a 45-mer
            contigs.append(np.concatenate([lut[w], lut[rng.integers(0, 4, 22)]]))          # site is the FIRST window
    contigs.append(lut[g[:22]])                                                             # too short
    contigs.append(np.zeros(0, np.uint8))                                                   # empty
    for i in range(GLEN):                                                                   # N at each offset
        w = lut[g].copy(); w[i] = ord("N")
        contigs.append(np.concatenate([lut[rng.integers(0, 4, 5)], w, lut[rng.integers(0, 4, 5)]]))
    lens = [len(c) for c in contigs]
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    asc = bytes(np.concatenate(contigs))
    guides = g.reshape(1, GLEN)
    exp = oracle_rows(asc, off, guides, k)
    got = gpu_rows(asc, off, guides, k)
    assert got == exp
    assert len(exp) >= 10


def test_contig_swarm_over_65536():
    """SNP-genome shape: > 65536 contigs of 45 bp; records ordered by (id mod 65536, pos, id >> 16)."""
    rng = np.random.default_rng(9)
    nct = 70000
    lut = np.frombuffer(b"ACGT", dtype=np.uint8)
    codes = rng.integers(0, 4, (nct, 45)).astype(np.uint8)
    guides = rng.integers(0, 4, (3, GLEN)).astype(np.uint8); guides[:, 21:] = 2
    for c in list(range(0, nct, 997)) + [5, 65536 + 5, 69999]:
        gi = c % 3
        w = guides[gi].copy()
        w[int(rng.integers(0, 20))] ^= 1
        if c % 2:
            w = revcomp_codes(w)
        p = [0, 22, 7][c % 3]
        codes[c, p:p + GLEN] = w
    # identical (id mod 65536, pos) for contigs 5 and 65541, same guide and strand
    codes[65536 + 5] = codes[5]
    asc = bytes(lut[codes.reshape(-1)])
    off = (np.arange(nct + 1) * 45).astype(np.uint64)
    exp = oracle_rows(asc, off, guides, 4)
    got = gpu_rows(asc, off, guides, 4)
    assert got == exp
    import varscot_b200 as V
    text = V.PackedText.from_ascii(asc, off)
    with V.ScanContext(0) as ctx:
        ctx.upload(text)
        hits, _ = ctx.scan(guides, 4)
    _, coll = V.resolve_hits(hits, off)
    assert coll >= 1


@pytest.mark.parametrize("shards", [2, 3, 7])
def test_sharded_text_equals_whole(shards):
    case = make_case(seed=21, contig_lens=[50000, 45, 45, 45, 20000], n_guides=8, k=6)
    assert_same(case, shards=shards)


@pytest.mark.parametrize("use_source", [True, False])
@pytest.mark.parametrize("chunk_words,streamed,use_sparse", [(64, False, True), (64, True, True), (1000, True, False), (7, True, True),
                                                             (256, False, False), (1 << 22, True, True)])
def test_chunked_and_streamed_scan(chunk_words, streamed, use_sparse, use_source):
    """Pipeline chunks smaller than the text: chunk borders (halo word), per-chunk counters; masks uploaded dense, sparse, or
    computed on the device from the compact mask source (N-plane runs + contig-end plane)."""
    case = make_case(seed=61, contig_lens=[70000, 45, 45, 45, 0, 23, 40000], n_guides=9, k=6, pam="AG")
    assert_same(case, chunk_words=chunk_words, streamed=streamed, use_sparse=use_sparse, use_source=use_source)
    assert_same(case, shards=3, chunk_words=chunk_words, streamed=streamed, use_sparse=use_sparse, use_source=use_source)


def test_mask_source_dense_blocks_and_skipped_n_runs():
    """A contig-end plane with dense blocks (a swarm of 45-base contigs), N runs long enough for their bases to be skipped by
    the upload (>= 16384 words), and a chunk size that cuts through both: device-computed masks give the oracle's records."""
    rng = np.random.default_rng(77)
    lens = [600_000] + [45] * 6000 + [23, 22, 0, 46] + [30_000]
    asc = bytearray(rng.choice(np.frombuffer(b"ACGT", dtype=np.uint8), sum(lens)).tobytes())
    asc[20_000:20_000 + 540_000] = b"N" * 540_000          # 16875 words of N inside the first contig
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    # exact forward-strand sites: inside contigs, on the last window of a 45-mer (R4), and — never to be reported — across
    # contig borders and reaching into the N run
    sites = (100, 600_010, 601_045, 870_000, 899_000, 600_000 + 45 * 20 + 22, 600_000 + 45 * 10 - 10, 600_000 + 45 * 3000 - 22, 19_990)
    for p in sites:
        asc[p + 21:p + 23] = b"GG"
    import varscot_b200 as V
    guides = V.guide_codes([bytes(asc[p:p + 23]) for p in sites])
    case = type("Case", (), dict(ascii=bytes(asc), offsets=off, guides=guides, k=5, pam=None))
    text = V.PackedText.from_ascii(case.ascii, off)
    assert text.em_dense.sum() > 0 and text.nm_runs["count"].max() >= 16384
    n = assert_same(case, chunk_words=5000, streamed=True)
    assert n >= 6
    assert_same(case, chunk_words=1 << 20, streamed=False)
    assert_same(case, shards=2, chunk_words=4096, streamed=True, use_source=False)


def test_streamed_scan_leaves_text_resident():
    import varscot_b200 as V
    case = make_case(seed=62, contig_lens=[90000, 30000], n_guides=5, k=5)
    text = V.PackedText.from_ascii(case.ascii, case.offsets).pin()
    with V.ScanContext(0) as ctx:
        ctx.set_chunk_words(512)
        a, st = ctx.scan_text(text, case.guides, 5)
        assert st.n_chunks > 1 and st.h2d_bytes > text.n_words * 8
        b, st2 = ctx.scan(case.guides, 5)
        assert st2.h2d_bytes < 100000
    ra, _ = V.resolve_hits(a, case.offsets)
    rb, _ = V.resolve_hits(b, case.offsets)
    assert ra.tolist() == rb.tolist() and len(ra) > 0
    text.unpin()


def test_hit_buffer_overflow_and_fetch():
    import varscot_b200 as V
    case = make_case(seed=33, contig_lens=[200000], n_guides=16, k=8, plant=False)
    text = V.PackedText.from_ascii(case.ascii, case.offsets)
    with V.ScanContext(0) as ctx:
        ctx.upload(text)
        small, _ = ctx.scan(case.guides, 8, cap=4)          # forces VS_ERR_OVERFLOW + vs_scan_fetch
        big, _ = ctx.scan(case.guides, 8, cap=1 << 20)
    assert len(small) == len(big) > 4
    a, _ = V.resolve_hits(small, case.offsets)
    b, _ = V.resolve_hits(big, case.offsets)
    assert a.tolist() == b.tolist()
    exp = oracle_rows(case.ascii, case.offsets, case.guides, 8)
    assert [(x[0], x[3], x[1], x[2], x[4]) for x in a.tolist()] == [e[:5] for e in exp]


def test_repeat_scan_is_deterministic_after_resolve():
    import varscot_b200 as V
    case = make_case(seed=40, contig_lens=[100000], n_guides=10, k=6)
    text = V.PackedText.from_ascii(case.ascii, case.offsets)
    with V.ScanContext(0) as ctx:
        ctx.upload(text)
        r = []
        for _ in range(3):
            hits, _ = ctx.scan(case.guides, 6)
            r.append(V.resolve_hits(hits, case.offsets)[0].tolist())
    assert r[0] == r[1] == r[2]


def test_cli_sam_byte_identical_to_oracle_cli(tmp_path):
    """The drop-in executables against the oracle executable: same argv, byte-identical SAM."""
    case = make_case(seed=55, contig_lens=[80000, 45, 45, 0, 30000], n_guides=7, k=5, pam="AG")
    gfa, rfa = str(tmp_path / "genome.fa"), str(tmp_path / "guides.fa")
    names = ["chr1 some description", "chr1_100_REF", "chr1_100_ALT_122_A_C", "empty", "chr2"]
    write_fasta(gfa, names, case.ascii, case.offsets)
    ids = [f"guide{i}" for i in range(7)]
    gs = list(case.guide_strs)
    gs[3] = gs[3][:5] + "N" + gs[3][6:]          # N in a guide becomes A (R5)
    gs[4] = gs[4].lower()
    write_guides(rfa, ids, gs)
    idx = str(tmp_path / "idx" / "genome")
    os.makedirs(os.path.dirname(idx))
    r = subprocess.run([os.path.join(BIN, "bidir_index"), "-G", gfa, "-I", idx], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert "Number of sequences: 5" in r.stdout and "Index created successfully" in r.stdout
    for style in ("seqan", "samtools"):
        out, ref = str(tmp_path / f"out_{style}.sam"), str(tmp_path / f"ref_{style}.sam")
        r = subprocess.run([os.path.join(BIN, "bidir_mapping"), "-G", gfa, "-I", idx, "-R", rfa, "-M", "5", "-T", "2", "-P", "AG",
                            "-O", out, "--md-style", style], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        assert "Reads loaded (total: 7)." in r.stdout and "Index loaded." in r.stdout
        o = subprocess.run([os.path.join(ROOT, "oracle", "oracle_bidir_mapping"), "-G", gfa, "-R", rfa, "-M", "5", "-P", "AG", "-O", ref,
                            "--md-style", style], capture_output=True, text=True)
        assert o.returncode == 0, o.stderr
        a, b = open(out, "rb").read(), open(ref, "rb").read()
        assert len(b) > 0
        assert a == b
    # without a cached index the mapper packs the FASTA itself
    out2 = str(tmp_path / "out2.sam")
    r = subprocess.run([os.path.join(BIN, "bidir_mapping"), "-G", gfa, "-I", str(tmp_path / "nonexistent"), "-R", rfa, "-M", "5", "-P", "AG",
                        "-O", out2], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert open(out2, "rb").read() == open(str(tmp_path / "out_seqan.sam"), "rb").read()


def test_config1_shape_50mbp():
    """BASELINE config 1 shape: one 50 Mbp contig with N runs + a 20k-contig SNP swarm, 10 guides, k <= 4."""
    rng = np.random.default_rng(1)
    lut = np.frombuffer(b"ACGT", dtype=np.uint8)
    n = 50_000_000
    asc = lut[rng.integers(0, 4, n).astype(np.uint8)]
    for s in (0, n // 2, n - 10000):
        asc[s:s + 10000] = ord("N")
    guides = rng.integers(0, 4, (10, GLEN)).astype(np.uint8); guides[:, 21:] = 2
    for g in range(10):
        for j in range(12):
            w = guides[g].copy()
            nm = j % 6
            if nm:
                idx = rng.choice(GLEN, nm, replace=False); w[idx] = (w[idx] + 1) % 4
            if j % 2:
                w = revcomp_codes(w)
            p = int(rng.integers(20000, n - 20000))
            asc[p:p + GLEN] = lut[w]
    # SNP swarm: 10k SNVs -> REF + ALT 45-mers cut from the genome
    pos = np.sort(rng.integers(30000, n - 30000, 10000))
    swarm = []
    for p in pos:
        ref = asc[p - 22:p + 23].copy(); alt = ref.copy()
        alt[22] = lut[(int(np.where(lut == (alt[22] if alt[22] != ord("N") else ord("A")))[0][0]) + 1) % 4]
        swarm += [ref, alt]
    asc_all = np.concatenate([asc] + swarm)
    lens = [n] + [45] * len(swarm)
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    exp = oracle_rows(bytes(asc_all), off, guides, 4)
    got = gpu_rows(bytes(asc_all), off, guides, 4)
    assert got == exp
    assert len(exp) >= 60


def test_candidate_store_regrow_and_dense_hits():
    """Low-complexity text: every window is a forward candidate (8x the sized-for density) and every one is a hit."""
    import varscot_b200 as V
    n = 1_200_000
    asc = b"G" * n
    off = np.array([0, n], dtype=np.uint64)
    guides = np.full((1, GLEN), 2, dtype=np.uint8)
    text = V.PackedText.from_ascii(asc, off)
    with V.ScanContext(0) as ctx:
        ctx.set_chunk_words(8192)
        ctx.upload(text)
        hits, st = ctx.scan(guides, 0, cap=16)
    assert st.redo_chunks > 0
    assert st.n_cand_fwd == n - 22 and st.n_cand_rev == 0
    assert len(hits) == n - 22
    assert np.array_equal(np.sort(hits["pos"]), np.arange(n - 22, dtype=np.uint32))
    assert (hits["info"] == 0).all()


def test_map_packed_multi_device_equals_single():
    """vs_map_packed shards the text over every visible GPU (one host thread + context each) — same records."""
    import varscot_b200 as V
    nd = V.device_count()
    case = make_case(seed=71, contig_lens=[300000, 45, 45, 200000], n_guides=12, k=6)
    text = V.PackedText.from_ascii(case.ascii, case.offsets)
    a, _ = V.map_packed(text, case.guides, 6, devices=[0])
    b, st = V.map_packed(text, case.guides, 6, devices=list(range(nd)) if nd > 1 else [0, 0, 0])
    ra, _ = V.resolve_hits(a, case.offsets)
    rb, _ = V.resolve_hits(b, case.offsets)
    assert ra.tolist() == rb.tolist() and len(ra) > 0
    exp = oracle_rows(case.ascii, case.offsets, case.guides, 6)
    assert [(x[0], x[3], x[1], x[2], x[4]) for x in ra.tolist()] == [e[:5] for e in exp]


def test_pipeline_chain_bed_vcf_to_sam(tmp_path):
    """The front of the VARSCOT pipeline with our drop-ins only (VARSCOT:260,274,296-314): fasta_writer -> guides,
    vcf_loader -> SNP genome, bidir_index + bidir_mapping on the reference and on the SNP genome; every file is compared
    with the oracle chain (oracle/vcf_oracle.py + oracle_bidir_mapping)."""
    from oracle import vcf_oracle as VO
    rng = np.random.default_rng(123)
    lut = "ACGT"
    seq = list("".join(rng.choice(list(lut), 60000)))
    guides_pos = [1000, 9000, 20000, 41000]
    bed_rows, vcf_rows = [], []
    for gi, p in enumerate(guides_pos):
        seq[p + 21:p + 23] = "GG"                                     # the on-target carries an NGG PAM
        strand = "+" if gi % 2 == 0 else "-"
        bed_rows.append(("chr1", p, p + 23, f"guide{gi}", 0, "+"))
        # an off-target copy elsewhere with 2 reference mismatches, one of which a variant repairs
        q = p + 3000
        w = seq[p:p + 23]
        for off in (3, 12):
            w[off] = lut[(lut.index(w[off]) + 1) % 4]
        seq[q:q + 23] = w
        vcf_rows.append((q + 12, seq[q + 12], seq[p + 12], "0|1" if gi % 2 else "1|1"))
    # unrelated variants, some close together
    for p in (500, 510, 530, 15000, 15040, 33333):
        vcf_rows.append((p, seq[p], lut[(lut.index(seq[p]) + 2) % 4], "0|1"))
    vcf_rows.sort()
    g, bed, vcf = str(tmp_path / "genome.fa"), str(tmp_path / "t.bed"), str(tmp_path / "v.vcf")
    s = "".join(seq)
    with open(g, "w") as f:
        f.write(">chr1\n" + "\n".join(s[i:i + 60] for i in range(0, len(s), 60)) + "\n")
    open(bed, "w").write("".join("\t".join(map(str, r)) + "\n" for r in bed_rows))
    open(vcf, "w").write("##fileformat=VCFv4.2\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\tS1\n" +
                         "".join(f"chr1\t{p + 1}\t.\t{r}\t{a}\t.\t.\t.\tGT\t{gt}\n" for p, r, a, gt in vcf_rows))
    vp = os.path.join(ROOT, "build", "variant_processing_build")
    guides_fa, flank_fa, snp_fa = str(tmp_path / "guides.fa"), str(tmp_path / "flank.fa"), str(tmp_path / "snp.fa")
    assert subprocess.run([os.path.join(vp, "fasta_writer"), guides_fa, flank_fa, bed, g]).returncode == 0
    assert subprocess.run([os.path.join(vp, "vcf_loader"), vcf, snp_fa, g, "0", "23", "1"], capture_output=True).returncode == 0
    exp_snp = str(tmp_path / "exp_snp.fa")
    VO.write_fasta(exp_snp, VO.vcf_loader(vcf, g))
    assert open(snp_fa).read() == open(exp_snp).read()
    total = 0
    for label, fa in (("ref", g), ("snp", snp_fa)):
        idx = str(tmp_path / f"{label}_idx")
        assert subprocess.run([os.path.join(BIN, "bidir_index"), "-G", fa, "-I", idx], capture_output=True).returncode == 0
        out, ref = str(tmp_path / f"{label}.sam"), str(tmp_path / f"{label}_oracle.sam")
        r = subprocess.run([os.path.join(BIN, "bidir_mapping"), "-G", fa, "-I", idx, "-R", guides_fa, "-M", "3", "-T", "1", "-O", out], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        o = subprocess.run([os.path.join(ROOT, "oracle", "oracle_bidir_mapping"), "-G", fa, "-R", guides_fa, "-M", "3", "-O", ref], capture_output=True, text=True)
        assert o.returncode == 0, o.stderr
        a = open(out, "rb").read()
        assert a == open(ref, "rb").read()
        total += a.count(b"\n")
        if label == "snp":
            # the repaired off-targets are found in ALT segments with one mismatch fewer than on the reference
            assert any(b"_ALT_" in l and b"NM:i:1" in l for l in a.splitlines())
    assert total >= 8
    # ... and the back of the pipeline (VARSCOT:332-337): bam_merger over the CUDA mapper's SAM files vs the oracle merger
    from oracle import merge_oracle as MO
    tus = str(tmp_path / "activity.txt")
    open(tus, "w").write("ID Sequence Score Dir\n" + "".join(f"guide{i} {'A' * 30} {1.5 + i} +\n" for i in range(4)))
    for mit in (0, 1):
        out_txt, fm_txt = str(tmp_path / f"result{mit}.txt"), str(tmp_path / f"fm{mit}.txt")
        r = subprocess.run([os.path.join(vp, "bam_merger"), out_txt, fm_txt, str(tmp_path / "ref.sam"), str(tmp_path / "snp.sam"), bed, g, snp_fa, tus,
                            "3", "23", "1", str(mit)], capture_output=True, text=True)
        assert r.returncode == 0, r.stdout + r.stderr
        exp_text, exp_fm = MO.bam_merger(str(tmp_path / "ref_oracle.sam"), str(tmp_path / "snp_oracle.sam"), bed, g, snp_fa, tus, 23, mit)
        assert open(out_txt).read() == exp_text and exp_text.count("\n") > 4
        if mit:
            assert open(fm_txt).read() == exp_fm


def rows_from_records(text, rec, offsets, guides, with_md=True):
    import varscot_b200 as V
    rows = []
    for r in rec:
        md = V.md_string(text, int(offsets[r["contig"]]) + int(r["pos"]), guides[r["guide"]], (int(r["flag"]) >> 4) & 1) if with_md else ""
        rows.append((int(r["guide"]), int(r["flag"]), int(r["contig"]), int(r["pos"]), int(r["mm"]), md))
    return rows


def gpu_rows_resolved(case, shards=1, streamed=True, use_source=True, chunk_words=None, hit_capacity=0, use_sink=False, threads=2):
    """The path of the executables: every shard's hits are resolved to (contig, pos) and sorted ON THE DEVICE
    (vs_scan_resolved), the host merges the lists (vs_merge_resolved)."""
    import varscot_b200 as V
    from varscot_b200 import _lib
    text = V.PackedText.from_ascii(case.ascii, case.offsets)
    if not use_source:
        text.em_code = None
    nw = text.n_words
    bounds = [nw * i // shards for i in range(shards + 1)]
    lists, stats = [], []
    for i in range(shards):
        if bounds[i + 1] <= bounds[i]:
            continue
        with V.ScanContext(0) as ctx:
            if chunk_words:
                ctx.set_chunk_words(chunk_words)
            if hit_capacity:
                ctx.set_option(_lib.VS_OPT_HIT_CAPACITY, hit_capacity)
            got = []
            sink = (lambda h, lo, hi: got.append(h.copy()) or 0) if use_sink else None
            if streamed:
                hits, st = ctx.scan_resolved(case.guides, case.k, pam=case.pam, text=text, first_word=bounds[i], n_words=bounds[i + 1] - bounds[i],
                                             cap=1 << 12, sink=sink)
            else:
                ctx.upload(text, bounds[i], bounds[i + 1] - bounds[i])
                hits, st = ctx.scan_resolved(case.guides, case.k, pam=case.pam, cap=1 << 12, sink=sink)
            if use_sink:
                hits = np.concatenate(got) if got else np.zeros(0, V.LOC_DT)
            # every list arrives sorted in emission-key order
            keys = (hits["info"].astype(np.uint64) >> np.uint64(7) << np.uint64(48)) | (hits["key"] & np.uint64((1 << 48) - 1))
            assert (np.diff(keys.astype(np.int64)) >= 0).all() if len(keys) > 1 and int(keys.max()) < 2 ** 63 else True
            lists.append(hits.copy())
            stats.append(st)
    rec, coll = V.merge_resolved(lists, threads=threads)
    return rows_from_records(text, rec, case.offsets, case.guides), stats, coll


@pytest.mark.parametrize("shards,streamed,use_source", [(1, True, True), (1, False, True), (3, True, True), (4, False, True), (2, True, False)])
def test_resolved_scan_equals_oracle(shards, streamed, use_source):
    case = make_case(seed=81, contig_lens=[50000, 45, 45, 45, 23, 22, 46, 20000] + [45] * 300 + [7000], n_guides=9, k=6, pam="AG")
    exp = oracle_rows(case.ascii, case.offsets, case.guides, case.k, case.pam)
    got, _, _ = gpu_rows_resolved(case, shards=shards, streamed=streamed, use_source=use_source, chunk_words=700)
    assert got == exp and len(exp) > 20


def test_resolved_scan_with_empty_contigs_uploads_the_offsets():
    """Empty contigs have no bit in the contig-end plane: the device notices (end-bit count) and the host's offsets are used."""
    case = make_case(seed=82, contig_lens=[0, 30000, 0, 0, 45, 0, 45, 23, 0, 9000, 0], n_guides=6, k=5)
    exp = oracle_rows(case.ascii, case.offsets, case.guides, case.k, case.pam)
    for shards, streamed in ((1, True), (1, False), (3, True)):
        got, _, _ = gpu_rows_resolved(case, shards=shards, streamed=streamed)
        assert got == exp and len(exp) > 5


def test_resolved_scan_over_65536_contigs_orders_ties_by_full_id():
    rng = np.random.default_rng(19)
    nct = 70000
    lut = np.frombuffer(b"ACGT", dtype=np.uint8)
    codes = rng.integers(0, 4, (nct, 45)).astype(np.uint8)
    guides = rng.integers(0, 4, (3, GLEN)).astype(np.uint8); guides[:, 21:] = 2
    for c in list(range(0, nct, 1499)) + [5, 65536 + 5]:
        w = guides[c % 3].copy()
        w[int(rng.integers(0, 20))] ^= 1
        codes[c, 7:7 + GLEN] = w
    codes[65536 + 5] = codes[5]                               # same (id mod 65536, pos), same guide and strand
    case = type("Case", (), dict(ascii=bytes(lut[codes.reshape(-1)]), offsets=(np.arange(nct + 1) * 45).astype(np.uint64), guides=guides, k=4, pam=None))
    exp = oracle_rows(case.ascii, case.offsets, case.guides, 4)
    got, _, coll = gpu_rows_resolved(case, shards=2)
    assert got == exp and coll >= 1


def test_resident_index_is_reused_and_rebuilt():
    """The first scan of a resident text builds the candidate index; scans with the same PAM set score it without
    extracting again; another -P, vs_index_drop or VS_OPT_KEEP_INDEX 0 rebuild it.  Results never change."""
    import varscot_b200 as V
    from varscot_b200 import _lib
    case = make_case(seed=83, contig_lens=[120000, 45, 45, 60000], n_guides=7, k=5)
    text = V.PackedText.from_ascii(case.ascii, case.offsets)
    exp = oracle_rows(case.ascii, case.offsets, case.guides, 5)
    exp_ag = oracle_rows(case.ascii, case.offsets, case.guides, 5, "AG")

    def rows(hits):
        rec, _ = V.resolve_hits(hits, case.offsets)
        return rows_from_records(text, rec, case.offsets, case.guides)

    with V.ScanContext(0) as ctx:
        ctx.set_chunk_words(900)
        ctx.upload(text)
        ctx.set_option(_lib.VS_OPT_BUCKET_INDEX, 0)             # the plain index only (its bucketed form has its own test)
        a, st_a = ctx.scan(case.guides, 5)
        b, st_b = ctx.scan(case.guides, 5)
        assert st_a.index_reused == 0 and st_a.extract_ms > 0
        assert st_b.index_reused == 1 and st_b.extract_ms == 0 and st_b.score_launches == 1
        assert (st_b.n_cand_fwd, st_b.n_blocks_fwd) == (st_a.n_cand_fwd, st_a.n_blocks_fwd)
        assert rows(a) == rows(b) == exp
        # fewer guides / another k against the same index
        c, st_c = ctx.scan(case.guides[:3], 3)
        assert st_c.index_reused == 1
        exp3 = oracle_rows(case.ascii, case.offsets, case.guides[:3], 3)
        rec, _ = V.resolve_hits(c, case.offsets)
        assert rows_from_records(text, rec, case.offsets, case.guides[:3]) == exp3
        d, st_d = ctx.scan(case.guides, 5, pam="AG")           # another PAM set: extracted again
        assert st_d.index_reused == 0 and rows(d) == exp_ag
        e, st_e = ctx.scan(case.guides, 5, pam="AG")
        assert st_e.index_reused == 1 and rows(e) == exp_ag
        ctx.drop_index()
        f, st_f = ctx.scan(case.guides, 5, pam="AG")
        assert st_f.index_reused == 0 and rows(f) == exp_ag
        ctx.set_option(_lib.VS_OPT_KEEP_INDEX, 0)
        for _ in range(2):
            g, st_g = ctx.scan(case.guides, 5)
            assert st_g.index_reused == 0 and rows(g) == exp
        ctx.set_option(_lib.VS_OPT_KEEP_INDEX, 1)
        ctx.upload(text, 0, text.n_words // 2)                  # a new upload drops the index
        h, st_h = ctx.scan(case.guides, 5)
        assert st_h.index_reused == 0 and len(h) < len(a)


@pytest.mark.parametrize("k,pam,n_guides", [(0, None, 5), (1, "AG", 40), (2, None, 7), (3, "TT", 33), (4, None, 130), (5, "AG", 9), (6, None, 100), (7, "CC", 12), (8, None, 36)])
def test_bucketed_index_equals_oracle(k, pam, n_guides):
    """The second scan of a resident text regroups the candidate index by PAM kind + the four bases next to the PAM
    (vs_bucket.cuh) and scores it with per-bucket mismatch budgets: same records as the oracle for every k, with the guide
    counts exercising full and 4-guide segments of every class, last windows, N runs, several shards."""
    import varscot_b200 as V
    from varscot_b200 import _lib
    case = make_case(seed=700 + k, contig_lens=[60000, 45, 45, 45, 23, 22, 46, 20000] + [45] * 200 + [9000], n_guides=n_guides, k=k, pam=pam,
                     guide_pam=(pam if pam in ("AG",) else "GG"))
    text = V.PackedText.from_ascii(case.ascii, case.offsets)
    exp = oracle_rows(case.ascii, case.offsets, case.guides, k, pam)
    for shards in (1, 3):
        lists = []
        nw = text.n_words
        for i in range(shards):
            w0, w1 = nw * i // shards, nw * (i + 1) // shards
            with V.ScanContext(0) as ctx:
                ctx.set_chunk_words(500)
                ctx.set_option(_lib.VS_OPT_BUCKET_INDEX, 2)           # whatever the guide count
                ctx.upload(text, w0, w1 - w0)
                h1, st1 = ctx.scan_resolved(case.guides, k, pam=pam)
                h2, st2 = ctx.scan_resolved(case.guides, k, pam=pam)        # builds and scores the bucketed index
                h3, st3 = ctx.scan_resolved(case.guides, k, pam=pam)
                assert (st1.index_reused, st2.index_reused, st3.index_reused) == (0, 2, 2)
                assert st2.index_build_ms > 0 and st3.index_build_ms == 0
                assert h1.tolist() == h2.tolist() == h3.tolist()            # sorted lists: identical, not just equal as sets
                lists.append(h3.copy())
        rec, _ = V.merge_resolved(lists)
        assert rows_from_records(text, rec, case.offsets, case.guides) == exp
    assert len(exp) > 0


def test_bucketed_index_many_guides_and_hit_buffer_regrow():
    import varscot_b200 as V
    from varscot_b200 import _lib
    case = make_case(seed=710, contig_lens=[90000], n_guides=1100, k=4, plant=False)
    rng = np.random.default_rng(5)
    codes = np.frombuffer(case.ascii, dtype=np.uint8).copy()
    lut = np.frombuffer(b"ACGT", dtype=np.uint8)
    for g in (0, 31, 32, 127, 128, 511, 1023, 1024, 1099):
        p = int(rng.integers(0, 90000 - GLEN))
        w = case.guides[g].copy()
        w[int(rng.integers(0, 23))] ^= 1
        if g % 2:
            w = revcomp_codes(w)
        codes[p:p + GLEN] = lut[w]
    case.ascii = bytes(codes)
    text = V.PackedText.from_ascii(case.ascii, case.offsets)
    exp = oracle_rows(case.ascii, case.offsets, case.guides, 4)
    with V.ScanContext(0) as ctx:
        ctx.set_option(_lib.VS_OPT_HIT_CAPACITY, 64)             # several guide passes over the bucketed index + regrowing
        ctx.upload(text)
        ctx.scan_resolved(case.guides, 4)
        hits, st = ctx.scan_resolved(case.guides, 4)
        assert st.index_reused == 2
    rec, _ = V.merge_resolved([hits])
    assert rows_from_records(text, rec, case.offsets, case.guides) == exp and len(exp) >= 9


@pytest.mark.parametrize("use_sink", [False, True])
def test_guide_super_chunks_with_a_small_hit_buffer(use_sink):
    """A device hit buffer far smaller than the hit count: the guides are scored in several passes over the resident index
    (config 5's mode); a sink receives every super-chunk as soon as it is sorted."""
    case = make_case(seed=84, contig_lens=[150000], n_guides=300, k=8, plant=False)
    exp = oracle_rows(case.ascii, case.offsets, case.guides, 8)
    assert len(exp) > 2000
    got, stats, _ = gpu_rows_resolved(case, streamed=True, hit_capacity=600, use_sink=use_sink, chunk_words=2000)
    assert got == exp
    assert stats[0].guide_passes > 2
    got2, stats2, _ = gpu_rows_resolved(case, streamed=False, hit_capacity=6, use_sink=use_sink)      # forces regrowing as well
    assert got2 == exp and stats2[0].redo_chunks > 0


def test_two_contexts_on_one_device_with_different_guides():
    """Two contexts of the same device scanning at the same time, each with its own > 256 guides: the pattern tables are
    per context (no shared __constant__ table), so neither sees the other's guides."""
    import threading
    import varscot_b200 as V
    cases = [make_case(seed=90 + i, contig_lens=[60000], n_guides=300, k=3 + i) for i in range(2)]
    out = [None, None]

    def work(i):
        text = V.PackedText.from_ascii(cases[i].ascii, cases[i].offsets)
        with V.ScanContext(0) as ctx:
            ctx.set_chunk_words(300)
            rows = None
            for _ in range(3):
                hits, _ = ctx.scan_resolved(cases[i].guides, cases[i].k, text=text)
                rec, _ = V.merge_resolved([hits])
                r = rows_from_records(text, rec, cases[i].offsets, cases[i].guides)
                assert rows is None or rows == r
                rows = r
            out[i] = rows

    th = [threading.Thread(target=work, args=(i,)) for i in range(2)]
    for t in th: t.start()
    for t in th: t.join()
    for i in range(2):
        assert out[i] == oracle_rows(cases[i].ascii, cases[i].offsets, cases[i].guides, cases[i].k) and len(out[i]) > 0


def test_map_records_multi_device_equals_oracle():
    import varscot_b200 as V
    nd = V.device_count()
    case = make_case(seed=72, contig_lens=[300000, 45, 45, 200000], n_guides=12, k=6)
    text = V.PackedText.from_ascii(case.ascii, case.offsets)
    exp = oracle_rows(case.ascii, case.offsets, case.guides, 6)
    for devices in ([0], list(range(nd)) if nd > 1 else [0, 0, 0]):
        rec, coll, st = V.map_records(text, case.guides, 6, devices=devices, threads=3)
        assert rows_from_records(text, rec, case.offsets, case.guides) == exp and coll == 0


def test_reference_driver_script_runs_on_the_drop_ins(tmp_path):
    """The reference's OWN driver (VARSCOT_pipeline/VARSCOT:21-357, made parseable by oracle/ref_hook/build_ref.sh: two stray
    `then` lines removed, nothing else) runs unchanged on our six executables: a sandbox holds the script, a link to build/
    and a stand-in for the external TUSCAN tool; the final hit table equals the oracle chain's, with and without a VCF."""
    import shutil
    drv = os.path.join(ROOT, "oracle", "_ref", "VARSCOT")
    if not os.path.exists(drv):
        pytest.skip("oracle/_ref/VARSCOT absent: the upstream driver script is not part of this repository "
                    "(__graft_entry__.build() derives it when VARSCOT_REFERENCE names a VARSCOT checkout)")
    from oracle import merge_oracle as MO, vcf_oracle as VO
    rng = np.random.default_rng(321)
    lut = "ACGT"
    seq = list("".join(rng.choice(list(lut), 50000)))
    bed_rows, vcf_rows = [], []
    for gi, p in enumerate((1500, 12000, 30500)):
        seq[p + 21:p + 23] = "GG"
        bed_rows.append(("chr1", p, p + 23, f"guide{gi}", 0, "+"))
        q = p + 4000
        w = seq[p:p + 23]
        for off in (2, 9):
            w[off] = lut[(lut.index(w[off]) + 1) % 4]
        seq[q:q + 23] = w
        vcf_rows.append((q + 9, seq[q + 9], seq[p + 9], "0|1"))
    for p in (700, 720, 25000, 41000):
        vcf_rows.append((p, seq[p], lut[(lut.index(seq[p]) + 2) % 4], "1|1" if p == 25000 else "0|1"))
    vcf_rows.sort()
    sand = tmp_path / "sandbox"
    (sand / "lib" / "TUSCAN" / "TUSCAN model").mkdir(parents=True)
    shutil.copy(drv, sand / "VARSCOT")
    os.symlink(os.path.join(ROOT, "build"), sand / "build")
    # stand-in for lib/TUSCAN (external tool, out of scope): the activity table bam_merger reads (feature_matrix.h:206-230)
    (sand / "lib" / "TUSCAN" / "TUSCAN model" / "TUSCAN.py").write_text(
        "import sys\n"
        "a = sys.argv\n"
        "inp, out = a[a.index('-i') + 1], a[a.index('-o') + 1]\n"
        "ids = [l[1:].strip() for l in open(inp) if l.startswith('>')]\n"
        "open(out, 'w').write('ID Sequence Score Dir\\n' + ''.join(f'{i} {\"A\" * 30} {1.25 + n} +\\n' for n, i in enumerate(ids)))\n")
    g, bed, vcf = str(tmp_path / "genome.fa"), str(tmp_path / "t.bed"), str(tmp_path / "v.vcf")
    s = "".join(seq)
    open(g, "w").write(">chr1\n" + "\n".join(s[i:i + 60] for i in range(0, len(s), 60)) + "\n")
    open(bed, "w").write("".join("\t".join(map(str, r)) + "\n" for r in bed_rows))
    open(vcf, "w").write("##fileformat=VCFv4.2\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\tS1\tS2\n" +
                         "".join(f"chr1\t{p + 1}\t.\t{r}\t{a}\t.\t.\t.\tGT\t{gt}\t0|0\n" for p, r, a, gt in vcf_rows))
    idx = str(tmp_path / "refidx")
    assert subprocess.run([os.path.join(BIN, "bidir_index"), "-G", g, "-I", idx], capture_output=True).returncode == 0
    env = dict(os.environ, PATH=os.path.dirname(os.sys.executable) + ":" + os.environ.get("PATH", ""))
    for with_vcf in (True, False):
        out = str(tmp_path / f"result_{int(with_vcf)}.txt")
        tdir = str(tmp_path / f"tmp_{int(with_vcf)}")
        cmd = ["bash", str(sand / "VARSCOT"), "-b", bed, "-o", out, "-g", g, "-i", idx, "-m", "3", "-t", "2", "-T", tdir, "-v"]
        if with_vcf:
            cmd += ["-f", vcf, "-s", "0"]
        r = subprocess.run(cmd, capture_output=True, text=True, env=env, timeout=600)
        assert r.returncode == 0, r.stdout + r.stderr
        assert "Analysis finished" in r.stdout
        # the oracle chain on the same inputs (files the driver left in its temp dir serve as the oracle's inputs where the
        # producing stage is covered by its own test: guides FASTA, activity table)
        guides_fa, act = os.path.join(tdir, "t.fa"), os.path.join(tdir, "t_activity.txt")
        ref_sam = str(tmp_path / f"oracle_ref_{int(with_vcf)}.sam")
        o = subprocess.run([os.path.join(ROOT, "oracle", "oracle_bidir_mapping"), "-G", g, "-R", guides_fa, "-M", "3", "-O", ref_sam], capture_output=True, text=True)
        assert o.returncode == 0, o.stderr
        prefix = os.path.basename(out)[:-4]
        assert open(os.path.join(tdir, f"{prefix}_reference.sam"), "rb").read() == open(ref_sam, "rb").read()
        if with_vcf:
            cut = str(tmp_path / "cut.vcf")
            open(cut, "w").write("".join("\t".join(l.rstrip("\n").split("\t")[:10]) + "\n" if not l.startswith("##") else l for l in open(vcf)))
            snp_fa = str(tmp_path / "oracle_snp.fa")
            VO.write_fasta(snp_fa, VO.vcf_loader(cut, g))
            assert open(os.path.join(tdir, f"{prefix}.fa")).read() == open(snp_fa).read()
            snp_sam = str(tmp_path / "oracle_snp.sam")
            o = subprocess.run([os.path.join(ROOT, "oracle", "oracle_bidir_mapping"), "-G", snp_fa, "-R", guides_fa, "-M", "3", "-O", snp_sam], capture_output=True, text=True)
            assert o.returncode == 0, o.stderr
            assert open(os.path.join(tdir, f"{prefix}_snp.sam"), "rb").read() == open(snp_sam, "rb").read()
            exp_text, _ = MO.bam_merger(ref_sam, snp_sam, bed, g, snp_fa, act, 23, 0)
        else:
            exp_text, _ = MO.bam_merger_ref_only(ref_sam, bed, g, act, 23, 0)
        lines = exp_text.splitlines(keepends=True)
        # the driver's last step: header, then the rows sorted on column 4 (VARSCOT:355-357, `sort -t$'\\t' -k4,4`)
        srt = subprocess.run(["sort", "-t", "\t", "-k4,4"], input="".join(lines[1:]), capture_output=True, text=True).stdout
        assert open(out).read() == lines[0] + srt and len(lines) > 3


def test_eight_concurrent_mapper_processes(tmp_path):
    """parallel.py:17,86-90 runs up to 48 pipelines at once and every pipeline two mappers (VARSCOT:321-323): eight
    bidir_mapping processes started together spread over the visible devices (pid % n) and write identical SAM files."""
    case = make_case(seed=56, contig_lens=[200000, 45, 45, 90000], n_guides=20, k=5)
    gfa, rfa = str(tmp_path / "genome.fa"), str(tmp_path / "guides.fa")
    write_fasta(gfa, ["chr1", "chr1_10_REF", "chr1_10_ALT_32_A_C", "chr2"], case.ascii, case.offsets)
    write_guides(rfa, [f"g{i}" for i in range(20)], case.guide_strs)
    idx = str(tmp_path / "idx")
    assert subprocess.run([os.path.join(BIN, "bidir_index"), "-G", gfa, "-I", idx], capture_output=True).returncode == 0
    env = dict(os.environ, VARSCOT_VERBOSE="1")
    procs = [subprocess.Popen([os.path.join(BIN, "bidir_mapping"), "-G", gfa, "-I", idx, "-R", rfa, "-M", "5", "-T", "1", "-O", str(tmp_path / f"o{i}.sam")],
                              stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, env=env) for i in range(8)]
    outs = [p.communicate(timeout=600) for p in procs]
    assert all(p.returncode == 0 for p in procs), [o[1] for o in outs]
    ref = str(tmp_path / "ref.sam")
    o = subprocess.run([os.path.join(ROOT, "oracle", "oracle_bidir_mapping"), "-G", gfa, "-R", rfa, "-M", "5", "-O", ref], capture_output=True, text=True)
    assert o.returncode == 0, o.stderr
    want = open(ref, "rb").read()
    assert len(want) > 0
    for i in range(8):
        assert open(str(tmp_path / f"o{i}.sam"), "rb").read() == want
    import varscot_b200 as V
    devs = {int(l.split("device ")[1].split()[0]) for _, e in outs for l in e.splitlines() if "scanning on device " in l}
    assert len(devs) == min(8, V.device_count())


def test_empty_inputs():
    """Empty text, zero guides, text shorter than a window: no hits, no errors."""
    import varscot_b200 as V
    g = np.full((2, GLEN), 2, dtype=np.uint8)
    with V.ScanContext(0) as ctx:
        for asc, off in ((b"", [0]), (b"", [0, 0, 0]), (b"ACGTACGTAC", [0, 10]), (b"G" * 22, [0, 22])):
            text = V.PackedText.from_ascii(asc, np.array(off, dtype=np.uint64))
            hits, st = ctx.scan_text(text, g, 4)
            assert len(hits) == 0 and st.n_hits == 0
        text = V.PackedText.from_ascii(b"G" * 100, np.array([0, 100], dtype=np.uint64))
        hits, _ = ctx.scan_text(text, np.zeros((0, GLEN), dtype=np.uint8), 4)
        assert len(hits) == 0
        hits, _ = ctx.scan_text(text, g[:1], 0)
        assert len(hits) == 78
        with pytest.raises(V.VarscotError):
            ctx.scan(g, 9)
        with pytest.raises(V.VarscotError):
            ctx.scan(np.full((1, GLEN), 7, dtype=np.uint8), 4)


def _plant(text, p, codes):
    """Write 23 Dna codes at global position p of a PackedText (bases only; masks are untouched)."""
    for i, c in enumerate(codes):
        w, b = (p + i) >> 5, np.uint32(1) << np.uint32((p + i) & 31)
        for name, bit in (("hi", (c >> 1) & 1), ("lo", c & 1)):
            if bit:
                text.bases[name][w] |= b
            else:
                text.bases[name][w] &= ~b


def test_full_size_properties_config3():
    """BASELINE config 3 at FULL size (3.1 Gbp genome + 5 M variants, 100 guides, k <= 6), checked through
    size-independent properties: every reported hit is re-verified from the packed planes (PAM on the genome, exact
    mismatch count, no N, inside one contig, R4 on last windows), no hit is reported twice, every planted site is
    found with its exact mismatch count, and the forward / reverse hit totals sit where uniform-random text puts them."""
    import varscot_b200 as V
    from varscot_b200 import synth
    rng = np.random.default_rng(2024)
    g = synth.synth_genome(11, 3_100_000_000, 24, 0.05)
    s = synth.synth_variant_segments(g, 12, 5_000_000)
    text = synth.concat_texts(g, s)
    del g, s
    guides = synth.synth_guides(13, 100)
    k = 6
    # plant sites at scannable positions: guide copies with j mismatches outside the PAM, both strands
    valid_words = np.flatnonzero(text.masks["iv"] == 0)
    planted = {}
    for j in range(240):
        gi, mm, strand = j % 100, j % 7, (j // 7) % 2
        w = int(valid_words[rng.integers(0, len(valid_words))])
        if w + 2 >= text.n_words or text.masks["iv"][w + 1] != 0:
            continue
        p = w * 32 + int(rng.integers(0, 32))
        codes = guides[gi].copy()
        idx = rng.choice(20, mm, replace=False)
        codes[idx] = (codes[idx] + rng.integers(1, 4, mm)) % 4
        if strand:
            codes = revcomp_codes(codes)
        if any(abs(p - q) < 46 for q, _ in planted):
            continue
        _plant(text, p, codes)
        planted[(p, (gi << 8) | (strand << 7))] = mm
    text.pin()
    with V.ScanContext(0) as ctx:
        hits, st = ctx.scan_text(text, guides, k, cap=1 << 20)
    text.unpin()
    assert 300_000 < len(hits) < 700_000                     # ~4.5e5 expected for uniform-random text
    pos = hits["pos"].astype(np.int64)
    info = hits["info"]
    gi, strand, mm = (info >> 8).astype(np.int64), ((info >> 7) & 1).astype(np.int64), (info & 0xF).astype(np.int64)
    # no duplicates
    key = (pos << 16) | (gi << 1) | strand
    assert len(np.unique(key)) == len(key)
    # window masks: every hit starts at a scannable position
    assert ((text.masks["iv"][pos >> 5] >> (pos & 31).astype(np.uint32)) & 1).sum() == 0
    # re-verify every hit from the planes
    hi = np.concatenate([text.bases["hi"], np.zeros(2, np.uint32)])
    lo = np.concatenate([text.bases["lo"], np.zeros(2, np.uint32)])
    wh, wl = synth._gather(hi, pos, 23), synth._gather(lo, pos, 23)
    pat = np.where(strand[:, None] == 1, 3 - guides[gi][:, ::-1], guides[gi]).astype(np.uint64)
    ph = ((pat >> np.uint64(1)) & np.uint64(1)) << np.arange(23, dtype=np.uint64)[None, :]
    pl = (pat & np.uint64(1)) << np.arange(23, dtype=np.uint64)[None, :]
    ph, pl = ph.sum(axis=1).astype(np.uint64), pl.sum(axis=1).astype(np.uint64)
    diff = (wh ^ ph) | (wl ^ pl)
    popc = np.array([bin(int(x)).count("1") for x in diff], dtype=np.int64)
    assert (popc == mm).all() and (mm <= k).all()
    code = lambda i: (((wh >> np.uint64(i)) & np.uint64(1)) << np.uint64(1)) | ((wl >> np.uint64(i)) & np.uint64(1))
    fwd_ok = (code(21) == 2) & ((code(22) == 2) | (code(22) == 0))               # GG, GA
    rev_ok = (code(1) == 1) & ((code(0) == 1) | (code(0) == 3))                  # CC, TC
    assert np.where(strand == 1, rev_ok, fwd_ok).all()
    # R4: hits on last windows have <= K = 3 mismatches in positions 11..22
    lastw = ((text.masks["lw"][pos >> 5] >> (pos & 31).astype(np.uint32)) & 1) == 1
    h2 = np.array([bin(int(x) >> 11).count("1") for x in diff[lastw]], dtype=np.int64)
    assert lastw.sum() > 100 and (h2 <= k // 2).all()
    # recall: every planted site with <= k mismatches is reported with its exact count
    found = {(int(p), int(i) & ~0x7F): int(m) for p, i, m in zip(pos, info, mm)}
    assert len(planted) > 150
    for (p, gk), m in planted.items():
        assert found.get((p, gk)) == m, (p, gk, m)
    # strands are balanced on random text
    nf, nr = int((strand == 0).sum()), int((strand == 1).sum())
    assert abs(nf - nr) < 0.05 * len(hits)
