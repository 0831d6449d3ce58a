"""bench.py's ORCHESTRATION on CPU: the multi-rank hand-over, the phases (index resident / cold / end to end / resident genome /
config-4 block / config 5 with a sink), the JSON line and the parity check — everything of the GPU arm except the device.

TEST INFRASTRUCTURE ONLY.  The scan context is replaced, inside this test process, by a stand-in that answers every scan with
the oracle's records for the rank's shard (same list format as vs_scan_resolved: resolved, sorted); NCCL is replaced by gloo.
Nothing of this can be reached from bench.py itself or from the product: the product has no CPU path.  What the dry run
proves is that bench.py's Python around the scans is sound at world sizes 1 (with the shared-memory hand-over forced) and 2 —
the part no single-GPU run exercises and a failed 8-GPU session of round 2 stumbled over (a sequence number reused across
phases made rank 0 merge stale lists)."""
import json
import os
import sys

import numpy as np
import pytest
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _install_fakes(world, rank, port):
    """Patch varscot_b200 / bench inside THIS process: fake scan context, no page-locking, gloo collectives."""
    sys.path.insert(0, ROOT)
    import ctypes as C
    import torch
    import torch.distributed as dist
    import varscot_b200 as V
    from varscot_b200 import _lib, mapper, synth
    from oracle import oracle as O
    import bench

    class FakeStats:
        def __init__(self, **kw):
            self.total_ms = 1.0; self.score_ms = 0.6; self.resolve_ms = 0.1; self.extract_ms = 0.3; self.upload_ms = 0.5
            self.launches = 3; self.score_launches = 1; self.n_chunks = 1; self.redo_chunks = 0; self.guide_passes = 1
            self.n_blocks_fwd = 100; self.n_blocks_rev = 100; self.n_cand_fwd = 3000; self.n_cand_rev = 3000
            self.index_reused = 0; self.index_build_ms = 0.0; self.h2d_bytes = 1000; self.d2h_bytes = 100; self.n_hits = 0
            self.__dict__.update(kw)

    class FakeCtx:
        """Answers like vs_scan_resolved, from the oracle: the records of the window starts the shard owns."""

        def __init__(self, device=0):
            self.text = None; self.first = 0; self.words = 0
            self.keep = 1; self.bucket = 1; self.scans = 0; self.cache = {}

        def measure_int_peaks(self):
            return 1.8e13, 9e12

        def set_option(self, opt, value):
            if opt == _lib.VS_OPT_KEEP_INDEX:
                self.keep = value
            if opt == _lib.VS_OPT_BUCKET_INDEX:
                self.bucket = value

        def upload(self, text, first_word=0, n_words=None, **kw):
            self.text, self.first, self.words = text, first_word, text.n_words - first_word if n_words is None else n_words
            self.scans = 0

        def close(self):
            pass

        def _records(self, text, first, words, guides, k, pam):
            key = (id(text), first, words, guides.tobytes(), k, pam)
            if key not in self.cache:
                s0, s1 = first * 32, min(text.n_bases, (first + words) * 32)
                e = min(text.n_bases, s1 + 23)
                codes = synth.unpack_codes(text, s0, e - s0)
                off_all = text.offsets.astype(np.int64)
                inner = off_all[(off_all > s0) & (off_all < e)] - s0
                off = np.concatenate([[0], inner, [e - s0]]).astype(np.uint64)
                r = O.map_guides(codes, off, guides, k, pam=pam)
                gpos = off[r.contig].astype(np.int64) + r.pos.astype(np.int64) + s0
                own = gpos < s1
                gpos = gpos[own]
                contig = np.searchsorted(text.offsets.astype(np.int64), gpos, side="right") - 1
                pos = gpos - text.offsets.astype(np.int64)[contig]
                strand = ((r.flag[own] & 16) >> 4).astype(np.uint64)
                loc = np.zeros(len(gpos), dtype=V.LOC_DT)
                loc["key"] = (r.guide[own].astype(np.uint64) << np.uint64(49)) | (strand << np.uint64(48)) | \
                             ((contig.astype(np.uint64) & np.uint64(0xFFFF)) << np.uint64(32)) | pos.astype(np.uint64)
                loc["contig"] = contig
                loc["info"] = (r.guide[own].astype(np.uint32) << 8) | (strand.astype(np.uint32) << 7) | r.mm[own]
                self.cache[key] = loc[np.argsort(loc["key"], kind="stable")]
            return self.cache[key]

        def scan_resolved(self, guides, k, pam=None, text=None, first_word=0, n_words=None, cap=1 << 20, out=None, sink=None):
            g = np.ascontiguousarray(guides, dtype=np.uint8).reshape(-1, 23)
            if text is not None:
                self.upload(text, first_word, n_words)
            loc = self._records(self.text, self.first, self.words, g, k, pam)
            st = FakeStats(n_hits=len(loc))
            if text is None and self.keep and self.scans >= 1:
                st.index_reused = 2 if (self.bucket and self.scans >= 2 and len(g) >= 64) else 1
                st.extract_ms = 0.0
            self.scans = self.scans + 1 if self.keep else 0
            if sink is not None:
                if os.environ.get("VS_FAKE_FAIL_DENSE_RANK") == str(rank):
                    raise RuntimeError("injected failure of the dense pass")
                half = len(g) // 2                            # two deliveries, as two guide super-chunks would arrive
                gid = loc["info"] >> 8
                for lo, hi in ((0, half), (half, len(g))):
                    part = loc[(gid >= lo) & (gid < hi)].copy()
                    part["key"] -= np.uint64(lo) << np.uint64(49)
                    if len(part) and sink(part, lo, hi):
                        raise RuntimeError("sink aborted")
                st.guide_passes = 2
                return None, st
            if out is None:
                return loc.copy(), st
            out[: len(loc)] = loc
            return out[: len(loc)], st

    V.ScanContext = FakeCtx
    mapper.PackedText.pin = lambda self: self
    mapper.PackedText.unpin = lambda self: None
    L = _lib.lib()
    keep = []

    def fake_host_alloc(n):
        buf = (C.c_uint8 * max(int(n), 16))()
        keep.append(buf)
        return C.addressof(buf)

    L.vs_host_alloc = fake_host_alloc
    L.vs_host_register = lambda p, n: 0
    L.vs_host_unregister = lambda p: 0
    L.vs_host_free = lambda p: None
    bench.bind_to_gpu_numa = lambda local: 0

    def dist_setup():
        if world > 1:
            os.environ["MASTER_ADDR"] = "127.0.0.1"; os.environ["MASTER_PORT"] = str(port)
            dist.init_process_group("gloo", rank=rank, world_size=world)
        return world, rank, rank

    def barrier(w, local):
        if w > 1:
            dist.barrier()

    def all_reduce(x, w, local, op):
        if w == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64)
        dist.all_reduce(t, op=getattr(dist.ReduceOp, op))
        return float(t.item())

    bench.dist_setup, bench.barrier, bench.all_reduce = dist_setup, barrier, all_reduce
    return bench


def _run(rank, world, port, argv, q):
    os.environ["CUDA_VISIBLE_DEVICES"] = ""                    # no device for the run nor its child processes, on a GPU machine too
    os.environ["MASTER_PORT"] = str(port)                      # (HostExchange names its segments after it)
    os.environ["TORCHELASTIC_RUN_ID"] = f"dry{port}"
    if world == 1:
        os.environ["VARSCOT_BENCH_FORCE_EXCHANGE"] = "1"
    bench = _install_fakes(world, rank, port)
    import io
    import contextlib
    sys.argv = ["bench.py"] + argv
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        bench.main()
    if rank == 0:
        q.put(buf.getvalue().strip().splitlines()[-1])


def _spawn(world, argv):
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 33500 + (os.getpid() % 2000) + 7 * world + len(argv)
    procs = [ctx.Process(target=_run, args=(r, world, port, argv, q)) for r in range(world)]
    for p in procs:
        p.start()
    line = q.get(timeout=900)
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    return json.loads(line)


@pytest.mark.parametrize("world", [1, 2, 3, 8])
def test_bench_orchestration_config3_with_target_block(world):
    d = _spawn(world, ["--gpus", str(world), "--config", "3", "--scale", "0.0002", "--steps", "2", "--warmup", "3"])
    assert d["n_gpus"] == world and d["scaling"] == "strong" and d["metric"] == "guide_Gbp_per_s"
    assert d["parity"]["diff"] == 0 and d["parity"]["hits_gpu"] == d["parity"]["hits_cpu"] > 0
    assert d["parity"]["tail"]["diff"] == 0 and d["parity"]["tail"]["hits_gpu"] > 0 and d["target_cfg4"]["parity"]["tail"]["diff"] == 0
    assert d["e2e"]["value"] > 0 and d["e2e_resident_genome"]["records_equal_full_upload"]
    assert d["index"] == "bucketed" and d["value_cold"] > 0 and d["value_plain_index"] > 0 and d["index_lists_identical"] is True
    t = d["target_cfg4"]
    assert t["index_lists_identical"] is True
    assert t["guides"] == 1000 and t["parity"]["diff"] == 0 and t["parity"]["hits_gpu"] > 0 and t["e2e"]["value"] > 0
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic", "frac_yardstick"} <= set(d["roofline"])
    # the config-5 block runs in a child process on the single-GPU line only; here (no device) the child must fail WITHOUT taking
    # the main line with it, and say why
    if world == 1:
        assert "error" in d["dense_cfg5"] and "exit code" in d["dense_cfg5"]["error"], d["dense_cfg5"]
        assert "error" in d["cli_e2e"]                        # the executable has no device here either: the leg reports it, the line stands
    else:
        c5 = d["dense_cfg5"]                                  # N > 1: config 5 in the same processes, on the same shards
        assert c5["n_gpus"] == world and c5["config"]["workload"].startswith("cfg5") and c5["hits_per_step"] > 0 and c5["redo"] == 0
        assert c5["verification"]["per_guide_counts_equal_small_scan"] and c5["parity"]["diff"] == 0 and c5["rank0"]["first_delivery_sorted"]


def test_bench_dense_block_failure_on_one_rank_costs_only_the_block(monkeypatch):
    """A rank whose config-5 pass fails reports it through one all-reduce: the other ranks do not wait for it, the block says why,
    and the main line (config 3 + config-4 block) is intact."""
    monkeypatch.setenv("VS_FAKE_FAIL_DENSE_RANK", "1")
    d = _spawn(2, ["--gpus", "2", "--config", "3", "--scale", "0.0002", "--steps", "2", "--warmup", "3"])
    assert "error" in d["dense_cfg5"] and "another rank" in d["dense_cfg5"]["error"]
    assert d["parity"]["diff"] == 0 and d["e2e"]["value"] > 0 and d["target_cfg4"]["parity"]["diff"] == 0


def test_bench_dump_outputs_are_the_records_of_the_timed_scan(tmp_path):
    """--dump-outputs writes the records of the last timed step of `value` as float64 columns; the stand-in answers with the oracle's
    records, so they must be the oracle's records of the whole text, in emission order."""
    _spawn(1, ["--config", "3", "--scale", "0.0002", "--steps", "2", "--warmup", "3", "--no-cpu", "--no-target", "--no-dense", "--no-cli",
               "--dump-outputs", str(tmp_path)])
    sys.path.insert(0, ROOT)
    import bench
    from oracle import oracle as O
    core = bench.load_synth_core()
    text = core.build_workload(3_100_000_000, 5_000_000, 0.0002)
    r = O.map_guides(core.unpack_codes(text, 0, text.n_bases), text.offsets, core.synth_guides(13, 100), 6)
    assert len(r.guide) > 0 and np.load(tmp_path / "hits_total.npy").tolist() == [len(r.guide)]
    assert not (tmp_path / "hits_index.npy").exists()
    for f in ("guide", "flag", "contig", "pos", "mm"):
        a = np.load(tmp_path / f"hits_{f}.npy")
        assert a.dtype == np.float64 and (a == getattr(r, f)).all(), f


def test_bench_config5_steps_and_dump_outputs(tmp_path):
    """Config 5 times --steps passes after --warmup ones; --dump-outputs writes its per-guide counts and, per guide, evenly spaced
    entries of what the sink received: here (oracle records) a subset of the oracle's hits, of the size the byte budget allows."""
    d = _spawn(1, ["--config", "5", "--scale", "0.0005", "--guides", "200", "--steps", "3", "--warmup", "1", "--no-cpu",
                   "--dump-outputs", str(tmp_path)])
    assert d["steps"] == 3 and d["warmup"] == 1 and d["hits_per_step"] > 100
    sys.path.insert(0, ROOT)
    import bench
    from oracle import oracle as O
    core = bench.load_synth_core()
    text = core.build_workload(3_100_000_000, 5_000_000, 0.0005)
    r = O.map_guides(core.unpack_codes(text, 0, text.n_bases), text.offsets, core.synth_guides(15, 200), 8)
    counts = np.bincount(r.guide, minlength=200)
    assert (np.load(tmp_path / "hits_per_guide.npy") == counts).all() and np.load(tmp_path / "hits_total.npy").tolist() == [len(r.guide)]
    got = {f: np.load(tmp_path / f"hits_{f}.npy").astype(np.int64) for f in ("guide", "strand", "contig", "pos", "mm")}
    per_guide = (bench.DUMP_BYTES - 4096 - 8 * 200) // (8 * 5 * 200)
    assert (np.bincount(got["guide"], minlength=200) == np.minimum(counts, per_guide)).all()
    exp = set(zip(r.guide.tolist(), ((r.flag & 16) >> 4).tolist(), r.contig.tolist(), r.pos.tolist(), r.mm.tolist()))
    assert set(zip(*(got[f].tolist() for f in ("guide", "strand", "contig", "pos", "mm")))) <= exp


@pytest.mark.parametrize("world", [1, 2])
def test_bench_orchestration_config5_sink(world):
    d = _spawn(world, ["--gpus", str(world), "--config", "5", "--scale", "0.0005", "--guides", "200"])
    assert d["n_gpus"] == world and d["hits_per_step"] > 100 and d["redo"] == 0
    assert d["verification"]["per_guide_counts_equal_small_scan"] and d["parity"]["diff"] == 0
    assert d["rank0"]["guide_passes"] == 2 and d["rank0"]["first_delivery_sorted"]
