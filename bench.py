#!/usr/bin/env python
"""bench.py — guide·Gbp/s of the off-target scan (BASELINE.json metric) on 1..8 B200.

A step = one full scan of all guides (both strands, <= k mismatches, PAM on the genome) over the synthetic text of the
config: reference genome + variant haplotype segments ("SNP genome").  With N > 1 ranks ONE text is cut into N word
ranges by vs_shard_bounds (the partition north_star names; `--scaling weak` keeps round 1's one-text-per-rank mode); there
is no collective on the data path, the ranks' hit lists meet in host shared memory and rank 0 merges them.
  value      : whole-job guide·Gbp/s with the packed text AND the candidate index resident in HBM (the analogue of the
               reference's prebuilt FM index); timed with CUDA events on the library's stream from the first kernel to the
               last resolved + sorted hit in host memory (SURVEY.md 8d), max over ranks
  value_cold : the same with the index dropped before every step (extraction of the PAM-valid windows included)
  e2e        : same metric through the C-ABI call with HOST buffers, wall clock: H2D of the rank's packed shard + guides,
               extraction, scoring, hit resolution + sort on the device, D2H, hand-over to rank 0 and the merge into
               records in emission order (vs_merge_resolved) — every step
  e2e_resident_genome : the per-sample call of a batch (parallel.py:86-90): the reference genome stays resident, only the
               variant segments and the guides travel
  roofline   : the scoring kernel against the MEASURED alu-pipe LOP3 rate: `frac` = executed LOP3 / peak; the dense-scan
               yardstick of SURVEY.md 8d (4.0 LOP3 per guide·bp) is reported as `frac_yardstick`
  cpu_baseline / parity : the CPU oracle (a port: linear XOR/popcount scan, not SeqAn's FM index) on a bounded sample, and
               the hit-set diff of the merged GPU records against it
  target_cfg4 : config 4 (1000 guides, k <= 6, +AG) on the same text and ranks — north_star's target
`--impl reference` times the CPU oracle alone on the same text and sample (the reference binary needs SeqAn, absent here).
"""
from __future__ import annotations

import argparse
import ctypes as C
import datetime
import hashlib
import importlib.util
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

C_ALG = 4.0            # yardstick LOP3 per guide·bp (SURVEY.md 8d): 64 per 32 starts per guide per strand


def csa_ops(n, init=False):
    """LOP3-class ops of popcount_planes<n, init> in vs_kernels.cuh: column compression, FA = 2 ops, HA = 2 ops."""
    ops, cols = 0, n
    for w in range(5):
        left = cols + (1 if init else 0)
        nxt = 0
        while left >= 2:
            left -= 2 if left >= 3 else 1
            ops += 2
            nxt += 1
        cols = nxt
    return ops


def score_ops(k):
    """(LOP3, LDS) k_score executes per (32-candidate block, guide) in stage A, and the extra of stage B."""
    pa = 23 if k >= 8 else 7 + 2 * k
    a = (csa_ops(pa) + 2, pa)
    b = (csa_ops(23 - pa, True) + 2, 23 - pa) if pa < 23 else (0, 0)
    return a, b


def bucketed_ops(guides, k, pam, keylen=8):
    """Mean (LOP3, LDS) k_score_bucketed executes per (32-candidate block, guide) in stage A on uniform text: a guide meets
    the buckets of a PAM kind with c = c_key + c_pam mismatches at the key positions, c_key ~ C(n, j) 3^j / 4^n over the 4^n
    buckets of the kind (n = keylen - 2 bases next to the PAM, whatever the guide), c_pam = its PAM against the kind's; the
    budget for the other 23 - keylen positions is K' = k - c (nothing is scored when K' < 0) and stage A loads
    PA' = min(23 - keylen, 9 + 2 K') of them (vs_bucket.cuh: bk_walk_slots)."""
    from math import comb
    kinds = [(2, 2), (2, 0)] + ([("ACGT".index(pam[0]), "ACGT".index(pam[1]))] if pam else [])
    n, rest = keylen - 2, 23 - keylen
    wk = [comb(n, j) * 3 ** j / 4.0 ** n for j in range(n + 1)]
    g = np.asarray(guides)
    lop = lds = 0.0
    for x, y in kinds:
        cp = (g[:, 21] != x).astype(int) + (g[:, 22] != y).astype(int)       # identical on both strands
        for j, w in enumerate(wk):
            kp = k - j - cp
            pa = np.minimum(rest, 9 + 2 * np.maximum(kp, 0))
            ops = np.array([csa_ops(int(a)) + 2 if q >= 0 else 0 for a, q in zip(pa, kp)], dtype=float)
            lop += w * ops.mean() / len(kinds)
            lds += w * np.where(kp >= 0, pa, 0).mean() / len(kinds)
    return lop, lds


CONFIGS = {
    # id: (description, genome bases, variants, guides, k, extra PAM, guide seed)
    1: ("cfg1: 10 guides vs 50 Mbp + 10k SNVs, <=4 mm", 50_000_000, 10_000, 10, 4, None, 3),
    2: ("cfg2: 100 guides vs 3.1 Gbp, reference only, <=4 mm", 3_100_000_000, 0, 100, 4, None, 13),
    3: ("cfg3: 100 guides vs 3.1 Gbp + 5M variants, <=6 mm", 3_100_000_000, 5_000_000, 100, 6, None, 13),
    4: ("cfg4: 1000 guides vs 3.1 Gbp + 5M variants, <=6 mm, NGG+NAG", 3_100_000_000, 5_000_000, 1000, 6, "AG", 14),
    5: ("cfg5: 10000 guides vs 3.1 Gbp + 5M variants, <=8 mm", 3_100_000_000, 5_000_000, 10000, 8, None, 15),
}


def load_synth_core():
    """varscot_b200/synth_core.py by path: numpy only, does not load the CUDA library (the reference arm uses it)."""
    spec = importlib.util.spec_from_file_location("vs_synth_core", os.path.join(ROOT, "varscot_b200", "synth_core.py"))
    m = importlib.util.module_from_spec(spec)
    sys.modules["vs_synth_core"] = m
    spec.loader.exec_module(m)
    return m


def config_dict(cfg, n_bases, n_contigs, scaling, scale):
    """The `config` object: identical in both arms."""
    desc, _, _, ng, k, pam, _ = cfg
    return {"workload": desc + (f" (scale {scale})" if scale != 1.0 else ""), "guides": ng, "k": k, "extra_pam": pam,
            "text_bases": int(n_bases), "contigs": int(n_contigs), "scaling": scaling,
            "l2": "inputs larger than L2 (126 MB): 2-bit text 0.25 B/base, candidate index 10 B per PAM-valid window"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled in the background (B200_PROFILING.md recipe)."""
    Q = "timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, device):
        self.rows = []
        self.device = device
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50", "-i", str(device)],
                                      stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.p = None

    def _read(self):
        for line in self.p.stdout:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 8:
                continue
            try:
                ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                self.rows.append((ts, float(f[1]), float(f[2]), float(f[3]), f[4], f[5], f[6], f[7]))
            except Exception:
                pass

    def stop(self, t0=None, t1=None):
        if not self.p:
            return None
        time.sleep(0.12)
        self.p.terminate()
        try:
            self.p.wait(timeout=2)
        except Exception:
            self.p.kill()
        rows = [r for r in self.rows if (t0 is None or r[0] >= t0 - 0.05) and (t1 is None or r[0] <= t1 + 0.05)]
        window = "timed"
        if not rows:
            rows, window = self.rows, "whole_run"
        if not rows:
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.device)],
                                     capture_output=True, text=True, timeout=10).stdout.strip().splitlines()[0]
                f = [x.strip() for x in out.split(",")]
                rows, window = [(time.time(), float(f[1]), float(f[2]), float(f[3]), f[4], f[5], f[6], f[7])], "after_timed"
            except Exception:
                return None
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[4 + i].lower().startswith("active") for r in rows)]
        sm = sorted(r[1] for r in rows)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": rows[0][2], "power_w_max": max(r[3] for r in rows),
                "reasons": reasons, "samples": len(rows), "window": window}


def bind_to_gpu_numa(local):
    """Pin this process to the CPUs next to its GPU (NVML affinity) BEFORE allocating page-locked buffers."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local)
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = [i for i in range(ncpu) if (words[i // 64] >> (i % 64)) & 1]
        allowed = set(os.sched_getaffinity(0))
        cpus = [c for c in cpus if c in allowed]
        if cpus:
            os.sched_setaffinity(0, cpus)
        return len(cpus)
    except Exception:
        return 0


def host_info():
    model = ""
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                model = line.split(":", 1)[1].strip()
                break
    except Exception:
        pass
    numa = 0
    try:
        numa = len([d for d in os.listdir("/sys/devices/system/node") if d.startswith("node") and d[4:].isdigit()])
    except Exception:
        pass
    return {"cpu_model": model, "cpus": len(os.sched_getaffinity(0)), "numa_nodes": numa}


def gpu_topology(txt=None):
    """`nvidia-smi topo -m` reduced to one line: link kinds between the GPUs and their CPU / NUMA affinity (VERDICT r1 item 2)."""
    try:
        import re
        import subprocess
        if txt is None:
            txt = subprocess.run(["nvidia-smi", "topo", "-m"], capture_output=True, text=True, timeout=20).stdout
        txt = re.sub(r"\x1b\[[0-9;]*m", "", txt)
        rows = [l.split("\t") for l in txt.splitlines() if l.startswith("GPU")]
        links, aff = set(), set()
        for r in rows:
            cells = [c.strip() for c in r[1:]]
            n_gpu = len(rows)
            links.update(c for c in cells[:n_gpu] if c and c != "X")
            aff.add(tuple(cells[n_gpu:n_gpu + 2]))
        return {"gpus": len(rows), "links": sorted(links), "cpu_numa_affinity": sorted("/".join(a) for a in aff)}
    except Exception:
        return None


def ncu_pipes():
    """ncu's own pipe loads of the scoring kernels from the committed round-2 captures (profiles/r2_*_summary.txt): what `roofline.frac`
    (executed stage-A LOP3 only) is a lower bound of.  Static evidence of an earlier run of the same kernels, quoted with its source."""
    out = {}
    want = {"alu_pct": "sm__inst_executed_pipe_alu.avg.pct_of_peak_sustained_active", "lsu_pct": "sm__inst_executed_pipe_lsu.avg.pct_of_peak_sustained_active",
            "smem_wavefronts_pct": "l1tex__data_pipe_lsu_wavefronts_mem_shared.sum.pct_of_peak_sustained_elapsed",
            "issue_pct": "smsp__issue_active.avg.pct_of_peak_sustained_active"}
    for label, name in (("k_score cfg3 x1.0", "r2_score_cfg3_summary.txt"), ("k_score cfg4 x1.0", "r2_score_cfg4_summary.txt"),
                        ("k_score_bucketed cfg4 x0.25", "r2_bucketed_cfg4_scale0.25_summary.txt")):
        try:
            d = {}
            for line in open(os.path.join(ROOT, "profiles", name)):
                f = line.split()
                for k, m in want.items():
                    if len(f) >= 2 and f[0] == m:
                        d[k] = float(f[1])
            if d:
                d["source"] = "profiles/" + name
                out[label] = d
        except Exception:
            pass
    return out or None


def dist_setup():
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local), timeout=datetime.timedelta(seconds=180))
    return world, rank, local


def barrier(world, local):
    if world > 1:
        import torch
        import torch.distributed as dist
        dist.barrier(device_ids=[local])
        torch.cuda.synchronize()


def all_reduce(x, world, local, op):
    if world == 1:
        return x
    import torch
    import torch.distributed as dist
    t = torch.tensor([x], dtype=torch.float64, device=f"cuda:{local}")
    dist.all_reduce(t, op=getattr(dist.ReduceOp, op))
    return float(t.item())


class HostExchange:
    """Hand-over of the ranks' sorted hit lists to rank 0 through POSIX shared memory ("merged on the host", north_star):
    every rank downloads its hits straight into its page-locked segment, publishes the counts with a sequence number, rank 0
    spins on the sequence numbers, merges, and publishes `done`.  The sequence number is one counter per object, advanced by
    every rank once per step (`begin`): steps of different measurement phases can never be mistaken for one another."""

    def __init__(self, V, world, rank, cap, pin=True, tag=None):
        from varscot_b200 import _lib
        self.V, self.world, self.rank, self.cap, self.pin = V, world, rank, cap, pin
        self.L = _lib.lib()
        tag = tag or (os.environ.get("MASTER_PORT", "0") + "_" + os.environ.get("TORCHELASTIC_RUN_ID", "x"))
        base = f"/dev/shm/varscot_bench_{tag}"
        self.paths = [f"{base}_{r}.bin" for r in range(world)]
        self.ctl_path = f"{base}_ctl.bin"
        self.n_ctl = 3 * world + 1                               # per rank: sequence number, count, second count; then `done`
        if rank == 0:
            np.zeros(self.n_ctl, dtype=np.int64).tofile(self.ctl_path)
        with open(self.paths[rank], "wb") as f:
            f.truncate(cap * 16)
        self.mine = np.memmap(self.paths[rank], dtype=V.LOC_DT, mode="r+", shape=(cap,))
        self.mine[:] = 0                                         # touch the pages before page-locking them
        if pin and self.L.vs_host_register(self.mine.ctypes.data, cap * 16) != 0:
            raise RuntimeError("vs_host_register failed")
        self.ctl = None
        self.others = None
        self.seq = 0

    def attach(self):
        """after a barrier: every segment exists"""
        self.ctl = np.memmap(self.ctl_path, dtype=np.int64, mode="r+", shape=(self.n_ctl,))
        if self.rank == 0:
            self.others = [self.mine if r == 0 else np.memmap(self.paths[r], dtype=self.V.LOC_DT, mode="r", shape=(self.cap,)) for r in range(self.world)]

    def begin(self):
        """every rank, once per step, in lockstep"""
        self.seq += 1
        return self.seq

    def publish(self, n, n2=0):
        self.ctl[3 * self.rank + 1] = n
        self.ctl[3 * self.rank + 2] = n2
        self.ctl[3 * self.rank] = self.seq                       # x86 keeps the store order; rank 0 reads the counts after the sequence number

    def collect(self, split=0):
        """rank 0: wait for every rank's list(s) of this step; split > 0: a second list starts at entry `split` of every segment"""
        lists = []
        deadline = time.time() + 120.0
        for r in range(self.world):
            while self.ctl[3 * r] < self.seq:
                if time.time() > deadline:
                    raise RuntimeError(f"rank {r} did not publish step {self.seq} within 120 s")
            if self.ctl[3 * r] != self.seq:
                raise RuntimeError(f"rank {r} is at step {int(self.ctl[3 * r])}, rank 0 at {self.seq}")
            lists.append(self.others[r][: int(self.ctl[3 * r + 1])])
            if split:
                lists.append(self.others[r][split: split + int(self.ctl[3 * r + 2])])
        return lists

    def done(self):
        self.ctl[3 * self.world] = self.seq

    def wait_done(self):
        deadline = time.time() + 120.0
        while self.ctl[3 * self.world] < self.seq:
            if time.time() > deadline:
                raise RuntimeError(f"rank 0 did not finish step {self.seq} within 120 s")

    def close(self):
        try:
            if self.pin:
                self.L.vs_host_unregister(self.mine.ctypes.data)
        except Exception:
            pass
        for p in ([self.paths[self.rank]] + ([self.ctl_path] if self.rank == 0 else [])):
            try:
                os.unlink(p)
            except OSError:
                pass


def cpu_sample(text, guides, k, pam, synth, target_s=12.0, max_bases=1 << 30):
    """Time the oracle (all host threads) on a bounded, word-aligned prefix of the text; return its records too."""
    from oracle import oracle as O
    probe = min(text.n_bases // 32 * 32, 16 << 20)
    codes = synth.unpack_codes(text, 0, probe)
    off = synth.slice_offsets(text, 0, probe)
    t = time.perf_counter()
    O.scan_count(codes, off, guides, k, pam)
    dt = max(time.perf_counter() - t, 1e-4)
    n = int(min(max_bases, text.n_bases, max(probe, probe * target_s / dt))) // 32 * 32
    codes = synth.unpack_codes(text, 0, n)
    off = synth.slice_offsets(text, 0, n)
    t = time.perf_counter()
    rec = O.map_guides(codes, off, guides, k, pam=pam)
    dt = time.perf_counter() - t
    return n, dt, rec, off, O.num_procs()


def parity_on_sample(rec_gpu, offsets, rec_cpu, off_cpu, n, start=0, end_is_real=False):
    """Hit-set diff (guide, strand, global position, NM) on the windows that start in [start, start + n): the oracle ran on that slice
    of the text.  A slice end that is not the text's end is an artificial contig end: the last 23 starts are left out there (a slice
    START cuts no window that starts inside the slice)."""
    hi = start + n - (0 if end_is_real else 23)
    gpos = offsets[rec_gpu["contig"]].astype(np.int64) + rec_gpu["pos"].astype(np.int64)
    sel = (gpos >= start) & (gpos < hi)
    gk = set(zip(rec_gpu["guide"][sel].tolist(), ((rec_gpu["flag"][sel] & 16) >> 4).tolist(), gpos[sel].tolist(), rec_gpu["mm"][sel].tolist()))
    opos = off_cpu[rec_cpu.contig].astype(np.int64) + rec_cpu.pos.astype(np.int64) + start
    osel = opos < hi
    ok = set(zip(rec_cpu.guide[osel].tolist(), ((rec_cpu.flag[osel] & 16) >> 4).tolist(), opos[osel].tolist(), rec_cpu.mm[osel].tolist()))
    return {"sample_bases": int(n), "hits_cpu": len(ok), "hits_gpu": len(gk), "diff": len(ok ^ gk)}


def parity_on_tail(rec_gpu, text, guides, k, pam, synth, max_bases):
    """The same diff on the LAST max_bases of the text — positions beyond 2^31 and, with variants, the swarm of 45-base contigs with
    ids far beyond 65535 — which the sample at the head of the text never reaches."""
    from oracle import oracle as O
    B = int(text.n_bases)
    s0 = max(0, B - int(max_bases)) // 32 * 32
    n = B - s0
    codes, off = synth.unpack_codes(text, s0, n), synth.slice_offsets(text, s0, n)
    rec = O.map_guides(codes, off, guides, k, pam=pam)
    d = parity_on_sample(rec_gpu, text.offsets, rec, off, n, start=s0, end_is_real=True)
    d["first_base"] = int(s0)
    return d


DUMP_BYTES = 64_000_000        # --dump-outputs: at most this much array data per run


def dump_arrays(out_dir, arrays, prefix=""):
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, prefix + name + ".npy"), np.asarray(a, dtype=np.float64))


def dump_records(out_dir, rec, prefix="", budget=DUMP_BYTES):
    """--dump-outputs: the records a caller receives (REC_DT, emission order) as float64 columns <prefix>hits_<field>.npy, exact for
    every field (u32 at most).  A list larger than the budget is replaced by a fixed sample (seed 0, indices sorted and written as
    <prefix>hits_index.npy); <prefix>hits_total.npy holds the full record count either way."""
    fields = ("guide", "flag", "contig", "pos", "mm")
    n = len(rec)
    cap = (budget - 4096) // (8 * (len(fields) + 1))
    arrays = {"hits_total": [n]}
    if n > cap:
        idx = np.sort(np.random.default_rng(0).choice(n, cap, replace=False))
        rec = rec[idx]
        arrays["hits_index"] = idx
    for f in fields:
        arrays["hits_" + f] = rec[f]
    dump_arrays(out_dir, arrays, prefix)


def run_reference(args, cfg, world, rank):
    """--impl reference: the CPU oracle port on the host cores (SeqAn's bidir_mapping cannot be built here).  Same text
    (seeds, scale) and the same kind of sample as the GPU arm's cpu_baseline; the product library is never loaded."""
    if rank != 0:
        return
    from oracle import oracle as O
    core = load_synth_core()
    desc, gbases, nvar, ng, k, pam, gseed = cfg
    guides = core.synth_guides(gseed, ng)
    text = core.build_workload(gbases, nvar, args.scale)
    budget_s = float(os.environ.get("VARSCOT_BENCH_BUDGET_S", "150")) / max(1, args.steps + args.warmup)
    probe = min(text.n_bases // 32 * 32, 8 << 20)
    t = time.perf_counter()
    O.scan_count(core.unpack_codes(text, 0, probe), core.slice_offsets(text, 0, probe), guides, k, pam)
    dt = max(time.perf_counter() - t, 1e-4)
    want = int(min(text.n_bases, 1 << 30, max(probe, probe * budget_s / dt))) // 32 * 32
    codes, off = core.unpack_codes(text, 0, want), core.slice_offsets(text, 0, want)
    for _ in range(args.warmup):
        O.scan_count(codes, off, guides, k, pam)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        O.scan_count(codes, off, guides, k, pam)
    dt = (time.perf_counter() - t0) / max(1, args.steps)
    val = ng * want / dt / 1e9
    cores = O.num_procs()
    sample = f"first {want} bases of the same text (seeds 11/12, scale {args.scale}), all {ng} guides, per step"
    scaling = "strong" if (world > 1 and args.scaling != "weak") else ("weak" if world > 1 else "single")
    print(json.dumps({
        "impl": "reference", "metric": "guide_Gbp_per_s", "value": val, "unit": "guide*Gbp/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "strong" if scaling != "weak" else "weak", "vs_baseline": None,
        "dtype": "u64 xor+popcount", "data": "synthetic", "config": config_dict(cfg, text.n_bases, len(text.offsets) - 1, scaling, args.scale),
        "cpu_baseline": {"value": val, "unit": "guide*Gbp/s", "cores": cores, "kind": "port", "sample": sample, **host_info()},
        "e2e": {"value": val, "unit": "guide*Gbp/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "CPU oracle port (linear 2-bit XOR/popcount scan, OpenMP, %d threads); the reference's SeqAn FM-index binary cannot be built: "
                "SeqAn 2.4.0rc2 is not vendored" % cores,
    }))


class Workload:
    """One config on this rank: pinned text, shard, context(s), hit buffers."""

    def __init__(self, V, text, shard_first, shard_words, local):
        self.V, self.text, self.first, self.words, self.local = V, text, shard_first, shard_words, local
        self.ctx = V.ScanContext(local)

    def close(self):
        self.ctx.close()


def measure(V, ctx, text, guides, k, pam, first, words, steps, warmup, world, local, hits_buf, exchange, n_total_bases, ng, host_threads,
            do_e2e=True, genome_words=None, keep_last=False):
    """value / value_cold / e2e (/ e2e_resident_genome) of one config on the given shard.  Returns a dict (rank 0: complete);
    keep_last: res["last_hits"] is a copy of the hit list of the last timed step of `value`."""
    from varscot_b200 import _lib
    res = {}
    units = float(ng) * n_total_bases                     # guide·bp per step over all ranks (strong: ONE text)
    ctx.upload(text, first, words)
    ctx.set_option(_lib.VS_OPT_KEEP_INDEX, 1)
    launches = 0
    # ---- index resident: its plain form (k_score), then its bucketed form (k_score_bucketed) -------------------------
    digests = {}
    for name, bucket in (("warm_plain", 0), ("warm", 1)):        # 1 = the library's default policy: bucketed where it pays
        ctx.set_option(_lib.VS_OPT_BUCKET_INDEX, bucket)
        build_ms = 0.0
        for _ in range(max(2, warmup)):
            hits, st = ctx.scan_resolved(guides, k, pam=pam, out=hits_buf)
            build_ms = max(build_ms, st.index_build_ms)
        barrier(world, local)
        dev = score = resolve = 0.0
        for _ in range(steps):
            hits, st = ctx.scan_resolved(guides, k, pam=pam, out=hits_buf)
            assert st.index_reused >= 1 and (bucket or st.index_reused == 1)
            dev += st.total_ms; score += st.score_ms; resolve += st.resolve_ms; launches += st.launches
        barrier(world, local)
        ms = all_reduce(dev / steps, world, local, "MAX")
        digests[name] = hashlib.blake2b(hits.tobytes(), digest_size=16).hexdigest()      # the sorted list of this rank's shard
        if keep_last and name == "warm":
            res["last_hits"] = hits.copy()                                             # hits_buf is reused by the next scans
        res[name] = {"ms": ms, "value": units / (ms * 1e-3) / 1e9, "score_ms": score / steps, "resolve_ms": resolve / steps, "launches": launches,
                     "score_launches": int(st.score_launches), "blocks": int(st.n_blocks_fwd + st.n_blocks_rev), "index_build_ms": build_ms,
                     "bucketed": bool(all_reduce(float(st.index_reused == 2), world, local, "MIN")),
                     "cands": int(st.n_cand_fwd + st.n_cand_rev), "hits": int(all_reduce(float(len(hits)), world, local, "SUM"))}
    # the two resident scans deliver byte-identical sorted lists on every rank (a full-size parity property: bucketed == plain)
    res["index_lists_identical"] = bool(all_reduce(float(digests["warm"] == digests["warm_plain"]), world, local, "MIN"))
    # ---- cold: the index is extracted again every step ------------------------------------------------
    res["launches"] = launches
    launches = 0
    ctx.set_option(_lib.VS_OPT_KEEP_INDEX, 0)
    for _ in range(2):
        ctx.scan_resolved(guides, k, pam=pam, out=hits_buf)
    barrier(world, local)
    dev = score = extract = 0.0
    for _ in range(steps):
        hits, st = ctx.scan_resolved(guides, k, pam=pam, out=hits_buf)
        dev += st.total_ms; score += st.score_ms; extract += st.extract_ms; launches += st.launches
    barrier(world, local)
    ms = all_reduce(dev / steps, world, local, "MAX")
    res["cold"] = {"ms": ms, "value": units / (ms * 1e-3) / 1e9, "score_ms": score / steps, "extract_ms": extract / steps, "chunks": int(st.n_chunks),
                   "score_launches": int(st.score_launches), "redo": int(st.redo_chunks)}
    res["launches"] += launches
    if not do_e2e:
        return res, None

    # ---- end to end: host buffers in, merged records out, every step --------------------------------------
    def e2e_loop(step_fn, n_steps):
        rec = coll = None
        for i in range(2):
            rec, coll = step_fn()
        barrier(world, local)
        t0 = time.perf_counter()
        for i in range(n_steps):
            rec, coll = step_fn()
        barrier(world, local)
        return (time.perf_counter() - t0) * 1e3 / n_steps, rec, coll

    stats = {}

    def full_step():
        if exchange is not None:
            exchange.begin()
        h, st2 = ctx.scan_resolved(guides, k, pam=pam, text=text, first_word=first, n_words=words, out=hits_buf)
        stats["st"] = st2
        if exchange is None:
            return V.merge_resolved([h], threads=host_threads)
        exchange.publish(len(h))
        out = (None, None)
        if exchange.rank == 0:
            out = V.merge_resolved(exchange.collect(), threads=host_threads)
            exchange.done()
        else:
            exchange.wait_done()
        return out

    e_ms, rec, coll = e2e_loop(full_step, steps)
    e_ms = all_reduce(e_ms, world, local, "MAX")
    st2 = stats["st"]
    res["e2e"] = {"value": units / (e_ms * 1e-3) / 1e9, "unit": "guide*Gbp/s", "ms_per_step": e_ms,
                  "h2d_bytes_per_step": int(all_reduce(float(st2.h2d_bytes), world, local, "SUM")),
                  "d2h_bytes_per_step": int(all_reduce(float(st2.d2h_bytes), world, local, "SUM")),
                  "rank0_device_ms": float(st2.total_ms), "rank0_upload_ms": float(st2.upload_ms),
                  "note": "vs_scan_resolved from pinned host buffers (H2D chunked, overlapped with extraction + scoring), hits resolved + sorted on the "
                          "device, D2H into shared memory, rank 0 merges all ranks' lists into records (vs_merge_resolved, %d threads); wall clock, max over ranks" % host_threads}
    ctx.set_option(_lib.VS_OPT_KEEP_INDEX, 1)
    ctx.set_option(_lib.VS_OPT_BUCKET_INDEX, 1)
    return res, (rec, coll)


def pick_canonical(h, key, idx):
    """h[idx] (a copy) of a key-sorted hit list, except that hits of equal key (contig ids equal modulo 2^16, same guide, strand and
    pos) arrive in no fixed order: a pick inside such a run takes the entry of the same rank in the run sorted by (contig, info)."""
    out = h[idx]
    tied = np.zeros(len(idx), dtype=bool)
    tied[idx > 0] |= key[idx[idx > 0] - 1] == out["key"][idx > 0]
    tied[idx < len(h) - 1] |= key[idx[idx < len(h) - 1] + 1] == out["key"][idx < len(h) - 1]
    for i in np.nonzero(tied)[0]:
        lo, hi = np.searchsorted(key, out["key"][i], "left"), np.searchsorted(key, out["key"][i], "right")
        run = h[lo:hi]
        out[i] = run[np.lexsort((run["info"], run["contig"]))[idx[i] - lo]]
    return out


def run_dense(args, cfg, V, synth, text, ctx, guides, first, words, world, rank, local, total_bases, all_cpus, t_gen, as_block=False):
    """Config 5 (10 000 guides, k <= 8: ~1.9e9 hits): passes through the end-to-end call with a sink, `--warmup` untimed ones, then
    `--steps` timed ones (as_block: one timed pass).  The guides are scored in super-chunks sized to the device hit buffer; every
    super-chunk is resolved + sorted on the device and handed to the host (here: counted per guide, spot-checked for order), so host
    memory stays O(super-chunk).
    Standalone (`--config 5`) rank 0 prints the line; as_block (the `dense_cfg5` block of a multi-GPU default line) rank 0 returns it.
    The device part runs without a collective inside and never raises: a rank that fails says so in ONE all-reduce after it, so that
    no rank is left waiting for another (standalone: every rank then raises; block: the block is {"error": ...})."""
    desc, gbases, nvar, ng, k, pam, gseed = cfg
    steps, warmup = (1, 0) if as_block else (args.steps, args.warmup)
    dump = bool(args.dump_outputs) and not as_block
    # --dump-outputs: per guide, up to `per_guide` of its delivered hits at evenly spaced ranks of its sorted list (the same entries
    # whatever the super-chunks: a guide's hits always arrive in one delivery)
    per_guide = max(1, (DUMP_BYTES // world - 4096 - 8 * ng) // (8 * 5 * ng))
    counts = np.zeros(ng, dtype=np.int64)
    box = {}

    def sink(h, lo, hi):
        """One delivery = the hits of guides [lo, hi), sorted; its key counts the guide from lo (bits 49..).  Per-guide counts come from
        the guide boundaries of the sorted list (binary searches on the strided key field: no pass over the 10^7..10^8 entries); every
        boundary is checked against the guide id stored in the record itself."""
        try:
            return sink_body(h, lo, hi)
        except Exception as e:                                  # (an exception cannot cross the C callback: abort the scan instead)
            box["error"] = repr(e)
            return 1

    def sink_body(h, lo, hi):
        t = time.perf_counter()
        key, info = h["key"], h["info"]
        b = np.searchsorted(key, np.arange(hi - lo + 1, dtype=np.uint64) << np.uint64(49))
        assert b[0] == 0 and b[-1] == len(h), "delivery holds guides outside its range"
        c = np.diff(b)
        nz = np.nonzero(c)[0]
        assert ((info[b[nz]] >> 8) == lo + nz).all() and ((info[b[nz + 1] - 1] >> 8) == lo + nz).all(), "guide boundaries of the delivery are off"
        counts[lo:hi] += c
        if box["chunks"] == 0:                                  # order spot check on the first delivery (a pass over its first 4 Mi entries)
            box["sorted"] = bool((np.diff(key[: 1 << 22].astype(np.int64)) >= 0).all())
        if dump:
            cs = c[nz]
            m = np.minimum(cs, per_guide)
            g = np.repeat(np.arange(len(nz)), m)
            j = np.arange(int(m.sum())) - np.repeat(np.cumsum(m) - m, m)
            box["sample"].append(pick_canonical(h, key, b[nz][g] + j * cs[g] // m[g]))
        box["chunks"] += 1; box["max_chunk"] = max(box["max_chunk"], len(h))
        box["host_s"] += time.perf_counter() - t
        return 0

    def one_pass():
        counts[:] = 0
        box.update(chunks=0, max_chunk=0, sorted=True, host_s=0.0, sample=[])
        t = time.perf_counter()
        _, st_ = ctx.scan_resolved(guides, k, pam=pam, text=text, first_word=first, n_words=words, sink=sink)
        return st_, (time.perf_counter() - t) * 1e3

    sampler = ClockSampler(local) if rank == 0 else None
    barrier(world, local)
    nv = 4
    err = None
    st = small = None
    dev_ms = wall_ms = 0.0
    t0_wall = time.time()
    try:
        for _ in range(warmup):
            one_pass()
        for _ in range(steps):
            st, w = one_pass()
            dev_ms += st.total_ms; wall_ms += w
        # verification scan of the first guides against the now resident index (same per-guide counts; parity with the oracle on a sample below)
        small, st_s = ctx.scan_resolved(guides[:nv], k, pam=pam, cap=1 << 22)
    except Exception as e:
        err = ("the sink refused a delivery: " + box["error"]) if "error" in box else repr(e)
    barrier(world, local)
    clocks = sampler.stop(t0_wall, time.time()) if sampler else None
    all_ok = all_reduce(0.0 if err else 1.0, world, local, "MIN") == 1.0
    if not all_ok:
        msg = f"config 5 failed on rank {rank}: {err}" if err else "config 5 failed on another rank"
        if not as_block:
            raise RuntimeError(msg)
        return {"error": msg} if rank == 0 else None
    ms = all_reduce(dev_ms / steps, world, local, "MAX")
    e_ms = all_reduce(wall_ms / steps, world, local, "MAX")
    hits_total = all_reduce(float(counts.sum()), world, local, "SUM")
    same_counts = bool((np.bincount((small["info"] >> 8).astype(np.int64), minlength=nv) == counts[:nv]).all())
    same_counts = all_reduce(1.0 if same_counts else 0.0, world, local, "MIN") == 1.0
    redo_total = int(all_reduce(float(st.redo_chunks), world, local, "SUM"))
    if dump:
        s = np.concatenate(box["sample"]) if box["sample"] else np.zeros(0, V.LOC_DT)
        dump_arrays(args.dump_outputs, {"hits_total": [counts.sum()], "hits_per_guide": counts, "hits_guide": s["info"] >> 8,
                                        "hits_strand": (s["info"] >> 7) & 1, "hits_contig": s["contig"],
                                        "hits_pos": s["key"] & np.uint64(0xFFFFFFFF), "hits_mm": s["info"] & 0x7F},
                    f"rank{rank}_" if world > 1 else "")
    if rank != 0:
        return None
    units = float(ng) * total_bases
    out = {"metric": "guide_Gbp_per_s", "value": units / (ms * 1e-3) / 1e9, "unit": "guide*Gbp/s", "n_gpus": world, "steps": steps, "warmup": warmup,
           "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u32 bit-sliced (LOP3)", "data": "synthetic",
           "config": config_dict(cfg, text.n_bases, text.n_contigs, "strong" if world > 1 else "single", args.scale),
           "value_note": "config 5 is measured in end-to-end passes (text from host buffers, hits to a host sink): value = mean CUDA-event time of the timed passes, e2e = their mean wall clock",
           "hits_per_step": int(hits_total), "hits_per_s": hits_total / (e_ms * 1e-3),
           "rank0": {"guide_passes": int(st.guide_passes), "redo": int(st.redo_chunks), "score_ms": float(st.score_ms), "extract_ms": float(st.extract_ms),
                     "resolve_sort_d2h_ms": float(st.resolve_ms), "sink_host_s": box["host_s"], "deliveries": box["chunks"], "largest_delivery": box["max_chunk"],
                     "first_delivery_sorted": box["sorted"], "hits": int(counts.sum())},
           "redo": redo_total, "gpu_launches": int(st.launches),
           "e2e": {"value": units / (e_ms * 1e-3) / 1e9, "unit": "guide*Gbp/s", "ms_per_step": e_ms, "h2d_bytes_per_step": int(st.h2d_bytes) * world,
                   "d2h_bytes_per_step": int(hits_total * 16)},
           "verification": {"guides": nv, "per_guide_counts_equal_small_scan": same_counts}, "clocks": clocks, "gen_s": t_gen, "host": host_info()}
    if not args.no_cpu:
        os.sched_setaffinity(0, all_cpus)
        n, dt, rec, off, cores = cpu_sample(text, guides[:nv], k, pam, synth, target_s=4.0 if as_block else 10.0, max_bases=min(1 << 28, words * 32))
        rec_g, coll = V.merge_resolved([small])
        out["parity"] = parity_on_sample(rec_g, text.offsets, rec, off, n)
        out["cpu_baseline"] = {"value": nv * n / dt / 1e9, "unit": "guide*Gbp/s", "cores": cores, "kind": "port",
                               "sample": f"first {n} bases, {nv} guides, one pass ({dt:.1f} s)", **host_info()}
    if as_block:
        for k_ in ("host", "gen_s", "vs_baseline", "higher_is_better", "data", "dtype", "steps", "warmup"):
            out.pop(k_, None)
        return out
    print(json.dumps(out))
    return out


def run_dense_child(args, timeout_s):
    """The `dense_cfg5` block of the default single-GPU line: config 5 at the same scale (10 000 guides, k <= 8, ~1.9e9 hits at full
    size) through `bench.py --config 5` in a CHILD process — after this process has released the GPU — so that whatever happens to it
    (error, time-out) costs the main line nothing but the block.  Returns the child's JSON line (bulky notes dropped) or {"error": ...}."""
    import signal
    env = {k_: v for k_, v in os.environ.items()
           if k_ not in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "LOCAL_WORLD_SIZE", "GROUP_RANK", "ROLE_RANK", "MASTER_ADDR", "MASTER_PORT", "TORCHELASTIC_RUN_ID")}
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--config", "5", "--gpus", "1", "--scale", repr(args.scale), "--steps", "1", "--warmup", "0"] + \
        (["--no-cpu"] if args.no_cpu else [])
    t = time.perf_counter()
    p = subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, env=env, start_new_session=True, cwd=ROOT)
    try:
        so, se = p.communicate(timeout=timeout_s)
    except subprocess.TimeoutExpired:
        try:
            os.killpg(p.pid, signal.SIGKILL)                 # exactly the session this call started
        except OSError:
            pass
        p.communicate()
        return {"error": f"child exceeded {timeout_s:.0f} s", "cmd": " ".join(cmd[1:])}
    wall = time.perf_counter() - t
    if p.returncode != 0:
        return {"error": f"child exit code {p.returncode}", "stderr_tail": se[-400:], "cmd": " ".join(cmd[1:])}
    try:
        d = json.loads(so.strip().splitlines()[-1])
    except Exception as e:
        return {"error": f"child line not parsed: {e!r}", "stdout_tail": so[-200:]}
    for k_ in ("host", "gen_s", "vs_baseline", "higher_is_better", "data", "dtype", "steps", "warmup"):
        d.pop(k_, None)
    d["child_wall_s"] = wall
    d["cmd"] = " ".join(["python"] + [os.path.basename(c) if c.endswith("bench.py") else c for c in cmd[1:]])
    return d


def run_cli_leg(V, text, guides, k, pam, threads):
    """`--cli`: the drop-in executable end to end, wall clock: bidir_mapping from the cached packed text (<prefix>.vsidx, written once
    by bidir_index) to the SAM file, one fresh process (CUDA context creation included), phases from its VARSCOT_VERBOSE lines."""
    import tempfile
    d = tempfile.mkdtemp(prefix="vs_cli_", dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
    try:
        prefix = os.path.join(d, "text")
        text.save(prefix)
        with open(prefix + ".vsnames", "w") as f:
            f.write("".join(f"ctg{i}\n" for i in range(text.n_contigs)))
        open(os.path.join(d, "genome.fa"), "w").write(">unused\nA\n")       # -G is only read when <prefix>.vsnames is missing
        with open(os.path.join(d, "guides.fa"), "w") as f:
            for i, g in enumerate(guides):
                f.write(f">g{i}\n{''.join('ACGT'[int(b)] for b in g)}\n")
        exe = os.path.join(ROOT, "build", "read_mapping_build", "bidir_mapping")
        cmd = [exe, "-G", os.path.join(d, "genome.fa"), "-I", prefix, "-R", os.path.join(d, "guides.fa"), "-M", str(k), "-T", str(threads),
               "-O", os.path.join(d, "out.sam")] + (["-P", pam] if pam else [])
        runs = []
        for _ in range(2):                                   # first process of the box pays driver initialisation; report both
            t = time.perf_counter()
            r = subprocess.run(cmd, capture_output=True, text=True, env=dict(os.environ, VARSCOT_VERBOSE="1", VARSCOT_GPUS="1"), timeout=120)
            wall = time.perf_counter() - t
            if r.returncode != 0:
                return {"error": r.stderr[-300:]}
            phases = [l.split(": ", 1)[1] for l in r.stderr.splitlines() if "wall:" in l or "upload+scan" in l]
            runs.append({"wall_s": wall, "phases": phases})
        n_rec = sum(1 for _ in open(os.path.join(d, "out.sam"), "rb"))
        return {"cmd": "bidir_mapping -G genome.fa -I <.vsidx cache> -R guides.fa -M %d -T %d -O out.sam" % (k, threads), "records": n_rec,
                "sam_bytes": os.path.getsize(os.path.join(d, "out.sam")), "vsidx_bytes": os.path.getsize(prefix + ".vsidx"), "runs": runs,
                "note": "one GPU (VARSCOT_GPUS=1), page cache warm, text cache in /dev/shm; wall clock of the whole process"}
    finally:
        import shutil
        shutil.rmtree(d, ignore_errors=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=3, choices=sorted(CONFIGS))
    ap.add_argument("--scale", type=float, default=1.0, help="shrink the text (quick runs only; invalid as a bench number)")
    ap.add_argument("--guides", type=int, default=0, help="override the number of guides")
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"],
                    help="strong (default): ONE text sharded over the ranks by vs_shard_bounds; weak: one text of the configured size per rank")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-target", action="store_true", help="skip the config-4 target block")
    ap.add_argument("--no-resident-genome", action="store_true")
    ap.add_argument("--no-dense", action="store_true", help="skip the dense_cfg5 block (config 5 in a child process; single-GPU default line only)")
    ap.add_argument("--cli", action="store_true", help="(default on the single-GPU config-3 line) the cli_e2e leg: the bidir_mapping executable from the .vsidx cache to the SAM file, wall clock")
    ap.add_argument("--no-cli", action="store_true", help="skip the cli_e2e leg")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step of `value` computed as DIR/<name>.npy (float64, at most 64 MB; "
                         "with several ranks every rank writes its shard's arrays as rank<r>_<name>.npy): its hit records in emission order; "
                         "config 5 its per-guide hit counts and a fixed sample of the hits its sink received")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if args.warmup < 3 and args.impl == "ours" and args.config != 5:      # (config 5's passes need no warm-up of a resident index)
        args.warmup = 3
    cfg = list(CONFIGS[args.config])
    if args.guides:
        cfg[3] = args.guides
    cfg = tuple(cfg)
    if args.impl == "reference":
        # the CPU arm needs no process group and no GPU: rank 0 (of the environment torchrun set) measures, the others leave at once
        run_reference(args, cfg, int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("RANK", "0")))
        return
    world, rank, local = dist_setup()
    all_cpus = os.sched_getaffinity(0)
    numa_cpus = bind_to_gpu_numa(local)

    import varscot_b200 as V
    from varscot_b200 import _lib, synth
    desc, gbases, nvar, ng, k, pam, gseed = cfg
    guides = synth.synth_guides(gseed, ng)
    strong = args.scaling == "strong" or world == 1
    t_gen = time.perf_counter()
    core_text = synth.core.build_workload(gbases, nvar, args.scale, 11 + (0 if strong else 1000 * rank), 12 + (0 if strong else 1000 * rank))
    text = synth.from_planes(core_text)
    t_gen = time.perf_counter() - t_gen
    genome_words = int(core_text.offsets[24] // 32) if nvar else text.n_words
    B, nw = text.n_bases, text.n_words
    first, words = 0, nw
    if strong and world > 1:
        sb = V.shard_bounds(nw, world)
        first, words = int(sb[rank]), int(sb[rank + 1] - sb[rank])
    text.pin()                                  # page-locked host buffers: what a caller of the C ABI hands in
    ctx = V.ScanContext(local)
    peak_lop3 = peak_lds = None
    if rank == 0:
        peak_lop3, peak_lds = ctx.measure_int_peaks()
    host_threads = max(1, min(16, len(all_cpus) - (world - 1)))      # rank 0 merges; the other ranks wait (one core each)

    def expected_hits(n_g, kk, n_pam, bases):
        """uniform-random text (SURVEY.md 8d): both strands, per PAM (1/16) P[Bin(21, 3/4) <= k]"""
        from math import comb
        p = sum(comb(21, j) * 0.75 ** j * 0.25 ** (21 - j) for j in range(kk + 1))
        return n_g * bases * 2.0 * n_pam / 16.0 * p

    B_mine = min(B - first * 32, words * 32)
    want = expected_hits(ng, k, 3 if pam else 2, B_mine)
    if args.config == 3 and not args.no_target and not args.guides:
        want = max(want, expected_hits(CONFIGS[4][3], CONFIGS[4][4], 3, B_mine))
    cap = 1 << 22
    while cap < 2.5 * want and cap < (1 << 26):
        cap <<= 1
    exchange = None
    if (world > 1 and strong) or os.environ.get("VARSCOT_BENCH_FORCE_EXCHANGE"):     # (the variable lets a one-GPU test exercise the shared-memory hand-over)
        exchange = HostExchange(V, world, rank, cap)
        barrier(world, local)
        exchange.attach()
        hits_buf = exchange.mine
    else:
        p = _lib.lib().vs_host_alloc(cap * 16)
        if not p:
            raise RuntimeError("vs_host_alloc failed")
        hits_buf = np.frombuffer((C.c_uint8 * (cap * 16)).from_address(p), dtype=V.LOC_DT, count=cap)
    total_bases = B if strong else all_reduce(float(B), world, local, "SUM")
    if args.config == 5:
        run_dense(args, cfg, V, synth, text, ctx, guides, first, words, world, rank, local, total_bases, all_cpus, t_gen)
        ctx.close()
        if exchange:
            barrier(world, local)
            exchange.close()
        return
    sampler = ClockSampler(local) if rank == 0 else None
    time.sleep(0.15)
    t0_wall = time.time()
    res, merged = measure(V, ctx, text, guides, k, pam, first, words, args.steps, args.warmup, world, local, hits_buf, exchange,
                          total_bases, ng, host_threads, do_e2e=not args.no_e2e, keep_last=bool(args.dump_outputs))
    clocks = sampler.stop(t0_wall, time.time()) if sampler else None
    if args.dump_outputs:
        rec_last, _ = V.merge_resolved([res.pop("last_hits")], threads=host_threads)
        dump_records(args.dump_outputs, rec_last, f"rank{rank}_" if world > 1 else "", DUMP_BYTES // world)
        del rec_last

    # ---- resident genome: only the variant segments (and the guides) travel per call ---------------------------
    e2e_rg = None
    if not args.no_e2e and not args.no_resident_genome and nvar and strong:
        gw0, gw1 = genome_words * rank // world, genome_words * (rank + 1) // world          # this rank's part of the genome ...
        sw = nw - genome_words
        sw0, sw1 = genome_words + sw * rank // world, genome_words + sw * (rank + 1) // world     # ... and of the variant segments
        gw0, gw1, sw0, sw1 = (x // 256 * 256 if x < nw else x for x in (gw0, gw1, sw0, sw1))
        if rank == world - 1:
            sw1 = nw
        ctx_g = V.ScanContext(local)
        ctx_g.upload(text, gw0, gw1 - gw0)
        half = cap // 2
        ctx_g.scan_resolved(guides, k, pam=pam, out=hits_buf[:half])                       # builds the genome's index once
        st_box = {}

        def rg_step():
            if exchange is not None:
                exchange.begin()
            # the resident genome and the uploaded segments are scanned at the same time (two contexts, two host threads)
            box = {}
            th = threading.Thread(target=lambda: box.update(g=ctx_g.scan_resolved(guides, k, pam=pam, out=hits_buf[:half])))
            th.start()
            b, sb_ = ctx.scan_resolved(guides, k, pam=pam, text=text, first_word=sw0, n_words=sw1 - sw0, out=hits_buf[half:])
            th.join()
            a, sa = box["g"]
            st_box["h2d"] = sa.h2d_bytes + sb_.h2d_bytes; st_box["d2h"] = sa.d2h_bytes + sb_.d2h_bytes
            if exchange is None:
                return V.merge_resolved([a, b], threads=host_threads)
            exchange.publish(len(a), len(b))                  # the two lists travel in one segment: [0, n_a) and [half, half + n_b)
            out = (None, None)
            if exchange.rank == 0:
                out = V.merge_resolved(exchange.collect(split=half), threads=host_threads)
                exchange.done()
            else:
                exchange.wait_done()
            return out

        for i in range(2):
            rg_step()
        barrier(world, local)
        t0 = time.perf_counter()
        for i in range(args.steps):
            rec_rg, _ = rg_step()
        barrier(world, local)
        rg_ms = all_reduce((time.perf_counter() - t0) * 1e3 / args.steps, world, local, "MAX")
        e2e_rg = {"value": float(ng) * total_bases / (rg_ms * 1e-3) / 1e9, "unit": "guide*Gbp/s", "ms_per_step": rg_ms,
                  "h2d_bytes_per_step": int(all_reduce(float(st_box["h2d"]), world, local, "SUM")),
                  "d2h_bytes_per_step": int(all_reduce(float(st_box["d2h"]), world, local, "SUM")),
                  "records_equal_full_upload": bool(rank != 0 or merged is None or (len(rec_rg) == len(merged[0]) and (rec_rg == merged[0]).all())),
                  "note": "per rank: its 1/N of the reference genome resident with its candidate index, its 1/N of the variant segments uploaded "
                          "and scanned per call (the per-sample call of parallel.py:86-90); records merged on rank 0 as in e2e"}
        ctx_g.close()

    # ---- config 4 target block (same text, 1000 guides, +AG) ---------------------------------------------------
    target = None
    if not args.no_target and args.config == 3 and not args.guides:
        c4 = CONFIGS[4]
        g4 = synth.synth_guides(c4[6], c4[3])
        tsteps = max(3, min(args.steps, 5))
        r4, merged4 = measure(V, ctx, text, g4, c4[4], c4[5], first, words, tsteps, 3, world, local, hits_buf, exchange, total_bases, c4[3], host_threads,
                              do_e2e=not args.no_e2e)
        if rank == 0:
            lop_a, lds_a = bucketed_ops(g4, c4[4], c4[5]) if r4["warm"]["bucketed"] else score_ops(c4[4])[0]
            target_ops = {"stage_a_lop3": lop_a, "stage_a_lds": lds_a}
            ex4 = lop_a * r4["warm"]["blocks"] * c4[3] / (r4["warm"]["score_ms"] * 1e-3)
            (lop_p4, _), _ = score_ops(c4[4])
            target = {"workload": c4[0], "guides": c4[3], "k": c4[4], "extra_pam": c4[5], "steps": tsteps,
                      "value": r4["warm"]["value"], "ms_per_step": r4["warm"]["ms"], "index_lists_identical": r4["index_lists_identical"], "value_cold": r4["cold"]["value"], "ms_per_step_cold": r4["cold"]["ms"],
                      "phase_ms_rank0": {"score": r4["warm"]["score_ms"], "resolve": r4["warm"]["resolve_ms"], "extract_cold": r4["cold"]["extract_ms"]},
                      "hits_per_step": r4["warm"]["hits"], "frac_executed": ex4 / peak_lop3, "executed_lop3_tlops": ex4 / 1e12,
                      "plain_index": {"value": r4["warm_plain"]["value"], "ms_per_step": r4["warm_plain"]["ms"], "score_ms": r4["warm_plain"]["score_ms"],
                                      "frac_executed": lop_p4 * r4["warm_plain"]["blocks"] * c4[3] / (r4["warm_plain"]["score_ms"] * 1e-3) / peak_lop3},
                      "index_build_ms_rank0": r4["warm"]["index_build_ms"], "ops_per_block_guide": target_ops,
                      "frac_note": "frac_executed counts the stage-A LOP3 of the adder trees only (a lower bound of the ALU-pipe load: the bucketed walk also "
                                   "issues one address update per slot and two blocks); ncu's own pipe loads of both kernels on this config: ncu_pipes",
                      "ncu_pipes": {k_: v for k_, v in (ncu_pipes() or {}).items() if "cfg4" in k_},
                      "e2e": r4.get("e2e"), "redo": r4["cold"]["redo"]}
            if not args.no_cpu and merged4 is not None:
                os.sched_setaffinity(0, all_cpus)
                n4, dt4, rec4, off4, cores4 = cpu_sample(text, g4, c4[4], c4[5], synth, target_s=10.0, max_bases=1 << 28)
                target["parity"] = parity_on_sample(merged4[0], text.offsets, rec4, off4, n4)
                target["parity"]["key16_collisions"] = int(merged4[1])
                target["parity"]["tail"] = parity_on_tail(merged4[0], text, g4, c4[4], c4[5], synth, 1 << 27)
                target["cpu_baseline"] = {"value": c4[3] * n4 / dt4 / 1e9, "unit": "guide*Gbp/s", "cores": cores4, "kind": "port",
                                          "sample": f"first {n4} bases, all {c4[3]} guides, one pass ({dt4:.1f} s)"}

    # ---- config 5 (10 000 guides, k <= 8, a hit sink) on the same text and ranks: at N > 1 in this process (one pass, no collective inside,
    # a failing rank reported by one all-reduce); at N = 1 in a child process after the GPU has been released (below) -------------------
    dense = None
    if world > 1 and strong and args.config == 3 and not args.no_dense and not args.guides:
        c5 = CONFIGS[5]
        dense = run_dense(args, c5, V, synth, text, ctx, synth.synth_guides(c5[6], c5[3]), first, words, world, rank, local, total_bases,
                          all_cpus, t_gen, as_block=True)
    if rank != 0:
        ctx.close()
        if exchange:
            barrier(world, local)
            exchange.close()
        return
    # ---- roofline of the dominant kernel (k_score) -----------------------------------------------------
    warm, cold, plain = res["warm"], res["cold"], res["warm_plain"]
    blocks = warm["blocks"]
    score_s = warm["score_ms"] * 1e-3
    B_local = min(B - first * 32, words * 32)             # bases whose window starts this rank owns
    (lop_p, lds_p), (lop_b, lds_b) = score_ops(k)
    bucketed = warm["bucketed"]                           # the library's policy decided (guide count, shard size)
    lop_a, lds_a = bucketed_ops(guides, k, pam) if bucketed else (lop_p, lds_p)
    executed = lop_a * blocks * ng / score_s             # stage A only: a lower bound (stage B runs for the few iterations that pass)
    lds = lds_a * blocks * ng / score_s
    yard = C_ALG * ng * B_local / score_s
    plain_s = plain["score_ms"] * 1e-3
    def dram_bytes(name):
        """dram__bytes_read.sum + dram__bytes_write.sum of one launch, from a committed ncu --set full summary (profiles/)."""
        try:
            rd = wr = None
            for line in open(os.path.join(ROOT, "profiles", name)):
                f = line.split()
                if len(f) >= 3 and f[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                    v = float(f[1]) * {"Mbyte": 1e6, "Gbyte": 1e9, "Kbyte": 1e3, "byte": 1.0}[f[2]]
                    rd, wr = (v, wr) if f[0].endswith("read.sum") else (rd, v)
            return rd + wr if rd is not None and wr is not None else None
        except Exception:
            return None
    # captures of round 2 (one launch each; the workload each was taken on is part of the name).  The number is only quoted as THIS run's traffic
    # when kernel and workload are the ones of this run: the full-size config-3 capture is of the plain-index kernel.
    captures = {"k_score cfg3 x1.0": dram_bytes("r2_score_cfg3_summary.txt"), "k_score cfg4 x1.0": dram_bytes("r2_score_cfg4_summary.txt"),
                "k_score_bucketed cfg4 x0.25": dram_bytes("r2_bucketed_cfg4_scale0.25_summary.txt")}
    same_workload = args.config == 3 and args.scale == 1.0 and world == 1
    traffic_plain = captures["k_score cfg3 x1.0"] if same_workload else None
    traffic = None if bucketed else traffic_plain
    hbm_peak = None
    try:
        hbm_peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]
    except Exception:
        pass
    hbm_alg = blocks * 192.0 / score_s / 1e9
    roof = {"bound": "int_alu", "kernel": "k_score_bucketed" if bucketed else "k_score", "achieved": executed / 1e12, "peak": peak_lop3 / 1e12, "unit": "Tlop3/s",
            "frac": executed / peak_lop3,
            "frac_note": "executed stage-A LOP3 of the scoring kernel (adder tree + 2 threshold ops per 32-candidate block and guide; the bucketed index scores "
                         "%.1f LOP3 / %.1f LDS per pair on average instead of the plain index's %d / %d) / measured alu-pipe LOP3 rate; a lower bound of the pipe load "
                         "(stage B, hit path, loop and segment overhead not counted); ncu pipe_alu / pipe_lsu of the same kernels: profiles/" % (lop_a, lds_a, lop_p, lds_p),
            "plain_index": {"kernel": "k_score", "score_ms": plain["score_ms"], "value": plain["value"], "ms_per_step": plain["ms"],
                            "frac": lop_p * blocks * ng / plain_s / peak_lop3, "frac_lds": lds_p * blocks * ng / plain_s / peak_lds,
                            "ops_per_block_guide": {"stage_a_lop3": lop_p, "stage_a_lds": lds_p}, "traffic": traffic_plain},
            "frac_yardstick": yard / peak_lop3,
            "yardstick_note": "dense-scan yardstick of SURVEY.md 8d: 4.0 LOP3 per guide*bp; the PAM-first index scores ~1/8 of the windows per strand, so this exceeds 1",
            "traffic": traffic, "algorithmic_bytes_per_launch": blocks * 192.0,
            "traffic_note": "dram bytes of one launch from the committed ncu --set full captures (profiles/r2_*_summary.txt); algorithmic = 192 B per block and launch. "
                            "The full-size config-3 capture of round 2 is of the plain-index kernel (plain_index.traffic); the bucketed kernel was captured on config 4 "
                            "at scale 0.25 only (traffic_captures), so its traffic on this workload is null, not guessed",
            "traffic_captures": captures,
            "ncu_pipes": ncu_pipes(),
            "hbm": {"achieved_gbs": hbm_alg, "peak_gbs": hbm_peak, "frac": (hbm_alg / hbm_peak) if hbm_peak else None,
                    "peak_source": "MEASURED_PEAKS.json hbm_gbs" if hbm_peak else "MEASURED_PEAKS.json absent"},
            "peak_source": "measured in this run by vs_measure_int_peaks (k_peak_lop3); MEASURED_PEAKS.json has no integer peak",
            "avg_launch_ms": warm["score_ms"] / max(1, warm["score_launches"]), "launches_per_step": warm["score_launches"],
            "ops_per_block_guide": {"stage_a_lop3": lop_a, "stage_a_lds": lds_a},
            "lds_words_per_s_T": lds / 1e12, "lds_peak_T": peak_lds / 1e12, "frac_lds": lds / peak_lds}
    scaling = "strong" if strong else "weak"
    out = {
        "metric": "guide_Gbp_per_s", "value": warm["value"], "unit": "guide*Gbp/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": warm["ms"], "higher_is_better": True, "scaling": scaling, "vs_baseline": None, "dtype": "u32 bit-sliced (LOP3)",
        "data": "synthetic", "config": config_dict(cfg, B, text.n_contigs, scaling if world > 1 else "single", args.scale),
        "value_note": "packed text AND candidate index resident in HBM (index = the PAM-valid windows of both strands, bucketed by PAM kind + the six bases next to "
                      "the PAM; built once per text and PAM set: the analogue of the reference's prebuilt FM index); first kernel -> resolved + sorted hits in host memory, "
                      "CUDA events, max over ranks",
        "index": "bucketed" if bucketed else "plain", "value_plain_index": plain["value"], "ms_per_step_plain_index": plain["ms"], "index_build_ms_rank0": warm["index_build_ms"],
        "index_lists_identical": res["index_lists_identical"],
        "index_lists_identical_note": "the scan of the resident plain index and the scan of the resident index in the form `value` used (bucketed where the "
                                      "policy says so) delivered byte-identical sorted hit lists on every rank: parity of the two kernels at full size",
        "value_cold": cold["value"], "ms_per_step_cold": cold["ms"],
        "value_cold_note": "the same with the index dropped before every step: extraction of the PAM-valid windows included",
        "layout": {"text_bases_per_gpu": int(B_local), "shard_words": int(words), "chunks": cold["chunks"], "cpus_bound_per_rank": numa_cpus,
                   "sharding": ("ONE text cut into %d word ranges by vs_shard_bounds, one per rank; no collective; hit lists merged by rank 0 in host shared memory" % world)
                               if strong else "one text per rank (weak), no collective",
                   "host_merge_threads": host_threads},
        "phase_ms_rank0": {"score": warm["score_ms"], "resolve_sort_d2h": warm["resolve_ms"], "extract_cold": cold["extract_ms"], "score_cold": cold["score_ms"]},
        "hits_per_step": warm["hits"], "candidates_rank0": warm["cands"], "gpu_launches": res["launches"], "redo": cold["redo"],
        "roofline": roof, "e2e": res.get("e2e"), "e2e_resident_genome": e2e_rg, "clocks": clocks, "gen_s": t_gen, "host": {**host_info(), "gpu_topology": gpu_topology()},
        "target_cfg4": target,
    }
    # ---- CPU baseline + hit-set diff of the MERGED records on a bounded sample -----------------------------
    if not args.no_cpu:
        os.sched_setaffinity(0, all_cpus)             # the CPU baseline gets every host core back
        n, dt, rec, off, cores = cpu_sample(text, guides, k, pam, synth)
        out["cpu_baseline"] = {"value": ng * n / dt / 1e9, "unit": "guide*Gbp/s", "cores": cores, "kind": "port",
                               "sample": f"first {n} bases of the same text, all {ng} guides, one pass ({dt:.1f} s); linear-scan oracle, not SeqAn", **host_info()}
        if merged is not None and merged[0] is not None:
            out["parity"] = parity_on_sample(merged[0], text.offsets, rec, off, n)
            out["parity"]["key16_collisions"] = int(merged[1])
            out["parity"]["tail"] = parity_on_tail(merged[0], text, guides, k, pam, synth, 1 << 28)
            out["parity"]["note"] = "records of the e2e path (all ranks merged on rank 0) vs the oracle; key16_collisions: records the reference's uint16 map key " \
                                    "(bidir_mapping.cpp:13) would have merged with another one — kept here (declared divergence R7)"
    ctx.close()
    if world == 1 and args.config == 3 and not args.no_dense:
        out["dense_cfg5"] = run_dense_child(args, float(os.environ.get("VARSCOT_BENCH_DENSE_TIMEOUT_S", "180")))
    else:
        out["dense_cfg5"] = dense                             # N > 1: measured in this process, above (None when skipped)
    if world == 1 and args.config == 3 and not args.no_cli:
        # the drop-in executable end to end (a fresh process per run: CUDA context, .vsidx mapped, scan, SAM): an error costs the block only
        try:
            text.unpin()
            out["cli_e2e"] = run_cli_leg(V, text, guides, k, pam, min(16, len(all_cpus)))
        except Exception as e:
            out["cli_e2e"] = {"error": repr(e)[:300]}
    print(json.dumps(out))
    if exchange:
        barrier(world, local)
        exchange.close()


def _shutdown():
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        try:
            import torch.distributed as dist
            if dist.is_initialized():
                dist.destroy_process_group()
        except Exception:
            pass


if __name__ == "__main__":
    try:
        main()
    except BaseException:
        # a rank that fails must take the job down at once: tearing the process group down gracefully would wait for the other
        # ranks, which are waiting for this one
        import traceback
        traceback.print_exc()
        sys.stdout.flush(); sys.stderr.flush()
        os._exit(1)
    _shutdown()
