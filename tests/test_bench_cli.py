"""bench.py keeps its contract: one JSON line with the required keys, for both arms.  The GPU arm runs a tiny copy of the
workload; the reference arm (CPU oracle) runs with a one-second budget."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
             "dtype", "data", "config", "e2e", "cpu_baseline"}


def test_reference_arm_line():
    env = dict(os.environ, VARSCOT_BENCH_BUDGET_S="2")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--config", "1", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0, r.stderr
    d = json.loads(r.stdout.strip().splitlines()[-1])
    assert BASE_KEYS <= set(d) and d["impl"] == "reference" and d["value"] > 0 and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]
    assert "workload" in d["config"]


@pytest.mark.gpu
def test_gpu_arm_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--config", "1", "--steps", "2", "--warmup", "3"],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr
    d = json.loads(r.stdout.strip().splitlines()[-1])
    assert BASE_KEYS | {"roofline", "gpu_launches", "clocks", "parity"} <= set(d)
    assert d["value"] > 0 and d["gpu_launches"] > 0 and d["scaling"] == "strong" and d["n_gpus"] == 1
    assert d["value_cold"] > 0 and d["value"] >= d["value_cold"] * 0.9 and d["redo"] == 0
    assert d["e2e_resident_genome"]["records_equal_full_upload"] and d["e2e_resident_genome"]["h2d_bytes_per_step"] < d["e2e"]["h2d_bytes_per_step"]
    assert d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] > 0 and d["e2e"]["value"] > 0
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(d["roofline"])
    assert d["parity"]["diff"] == 0 and d["cpu_baseline"]["value"] > 0 and d["roofline"]["frac"] < 1.2


@pytest.mark.gpu
def test_gpu_arm_shared_memory_handover_and_dense_mode():
    """The N > 1 hand-over (hits downloaded straight into a page-locked shared-memory segment, merged by rank 0) exercised on one
    GPU, and config 5's mode (one end-to-end pass with a hit sink, guide super-chunks) at a small scale."""
    env = dict(os.environ, VARSCOT_BENCH_FORCE_EXCHANGE="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--config", "1", "--steps", "2", "--warmup", "3", "--no-target"],
                       capture_output=True, text=True, timeout=900, env=env)
    assert r.returncode == 0, r.stderr
    d = json.loads(r.stdout.strip().splitlines()[-1])
    assert d["parity"]["diff"] == 0 and d["e2e"]["value"] > 0 and d["e2e_resident_genome"]["records_equal_full_upload"]
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--config", "5", "--scale", "0.004", "--guides", "600"],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr
    d = json.loads(r.stdout.strip().splitlines()[-1])
    assert d["hits_per_step"] > 10000 and d["redo"] == 0 and d["verification"]["per_guide_counts_equal_small_scan"]
    assert d["parity"]["diff"] == 0 and d["rank0"]["first_delivery_sorted"] and d["e2e"]["value"] > 0


@pytest.mark.gpu
def test_gpu_arm_dump_outputs_equal_oracle(tmp_path):
    """--dump-outputs: the records of the last timed scan, as written by the GPU arm, are the oracle's records of the same text."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--config", "3", "--scale", "0.001", "--steps", "2", "--warmup", "3",
                        "--no-cpu", "--no-e2e", "--no-target", "--no-dense", "--no-cli", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr
    assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 2
    sys.path.insert(0, ROOT)
    import numpy as np
    import bench
    from oracle import oracle as O
    core = bench.load_synth_core()
    text = core.build_workload(3_100_000_000, 5_000_000, 0.001)
    exp = O.map_guides(core.unpack_codes(text, 0, text.n_bases), text.offsets, core.synth_guides(13, 100), 6)
    assert len(exp.guide) > 0 and np.load(tmp_path / "hits_total.npy").tolist() == [len(exp.guide)]
    for f in ("guide", "flag", "contig", "pos", "mm"):
        assert (np.load(tmp_path / f"hits_{f}.npy") == getattr(exp, f)).all(), f


def test_dump_records_samples_a_large_list_the_same_way_every_time(tmp_path):
    sys.path.insert(0, ROOT)
    import numpy as np
    import bench
    from varscot_b200.mapper import REC_DT
    rec = np.zeros(1000, dtype=REC_DT)
    rec["guide"] = np.arange(1000) % 7; rec["contig"] = np.arange(1000) // 3; rec["pos"] = 4_000_000_000 - np.arange(1000); rec["mm"] = 2
    budget = 4096 + 48 * 100                                     # room for 100 records (5 columns + their indices)
    for d in ("a", "b"):
        bench.dump_records(str(tmp_path / d), rec, "rank1_", budget)
    idx = np.load(tmp_path / "a" / "rank1_hits_index.npy")
    assert len(idx) == 100 and (np.diff(idx) > 0).all() and np.load(tmp_path / "a" / "rank1_hits_total.npy").tolist() == [1000]
    for f in ("guide", "flag", "contig", "pos", "mm"):
        a = np.load(tmp_path / "a" / f"rank1_hits_{f}.npy")
        assert (a == rec[f][idx.astype(np.int64)]).all() and (a == np.load(tmp_path / "b" / f"rank1_hits_{f}.npy")).all()
    assert sum(os.path.getsize(p) for p in (tmp_path / "a").iterdir()) <= budget


def test_pick_canonical_ignores_the_order_of_equal_keys():
    """Hits of equal key may arrive in either order: the picks (and so config 5's dumped sample) must not depend on it."""
    sys.path.insert(0, ROOT)
    import numpy as np
    import bench
    from varscot_b200.mapper import LOC_DT
    h = np.zeros(12, dtype=LOC_DT)
    h["key"] = [1, 2, 5, 5, 5, 7, 8, 8, 9, 10, 11, 11]
    h["contig"] = np.arange(12) + 70000
    h["info"] = np.arange(12)
    other = h.copy()
    other[2:5] = h[2:5][::-1]                                    # the same list with its runs of equal keys in another order
    other[6:8] = h[6:8][::-1]
    other[10:12] = h[10:12][::-1]
    idx = np.array([0, 2, 3, 4, 7, 9, 11])
    a, b = bench.pick_canonical(h, h["key"], idx), bench.pick_canonical(other, other["key"], idx)
    assert (a == b).all() and sorted(a["contig"].tolist()) == sorted(h["contig"][idx].tolist())


def test_static_evidence_helpers():
    """The bench line quotes ncu's pipe loads and DRAM bytes from the committed captures and reduces `nvidia-smi topo -m` to one
    entry: both parsers against the files under profiles/ (no GPU, no nvidia-smi needed)."""
    sys.path.insert(0, ROOT)
    import bench
    pipes = bench.ncu_pipes()
    assert set(pipes) == {"k_score cfg3 x1.0", "k_score cfg4 x1.0", "k_score_bucketed cfg4 x0.25"}
    for d in pipes.values():
        assert 40 < d["alu_pct"] < 100 and 40 < d["lsu_pct"] < 100 and os.path.exists(os.path.join(ROOT, d["source"]))
    topo = bench.gpu_topology(open(os.path.join(ROOT, "profiles", "r2_box_8gpu.txt")).read())
    assert topo == {"gpus": 8, "links": ["NV18"], "cpu_numa_affinity": ["0-31/0"]}
    assert bench.host_info()["numa_nodes"] >= 0


def test_parity_windows_head_and_tail():
    """bench.py's hit-set diff on a slice of the text: the head sample (artificial END: its last 23 starts are left out) and the tail
    sample (artificial START: cuts nothing; real end) must both report 0 against records of the whole text, and notice a moved hit."""
    sys.path.insert(0, ROOT)
    import numpy as np
    import bench
    from oracle import oracle as O
    core = bench.load_synth_core()
    text = core.build_workload(3_100_000_000, 5_000_000, 0.0004)          # ~1.4 Mbases: genome + a swarm of variant segments
    guides = core.synth_guides(13, 60)
    full = O.map_guides(core.unpack_codes(text, 0, text.n_bases), text.offsets, guides, 6)
    rec = np.zeros(len(full.guide), dtype=[("guide", "<u4"), ("contig", "<u4"), ("pos", "<u4"), ("flag", "<u2"), ("mm", "u1")])
    for f in rec.dtype.names:
        rec[f] = getattr(full, f)
    n = text.n_bases // 2 // 32 * 32
    head = O.map_guides(core.unpack_codes(text, 0, n), core.slice_offsets(text, 0, n), guides, 6)
    d = bench.parity_on_sample(rec, text.offsets, head, core.slice_offsets(text, 0, n), n)
    assert d["diff"] == 0 and d["hits_gpu"] > 0
    t = bench.parity_on_tail(rec, text, guides, 6, None, core, text.n_bases // 3)
    assert t["diff"] == 0 and t["hits_gpu"] > 0 and t["first_base"] > 0 and t["first_base"] % 32 == 0
    gpos = text.offsets[rec["contig"]].astype(np.int64) + rec["pos"]
    i = int(np.nonzero(gpos >= t["first_base"])[0][0])
    rec["mm"][i] += 1
    assert bench.parity_on_tail(rec, text, guides, 6, None, core, text.n_bases // 3)["diff"] == 2
