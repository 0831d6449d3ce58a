#!/usr/bin/env python
"""Wall time of vs_map_records on a text beyond 4 Gbases, next to the config-3 size as the control (run on the GPU box).

The large text is a 5.5 Gbase synthetic genome plus the variant segments of 5 M variants (~5.9 Gbases): on one GPU it is
scanned as two shards one after the other, on several GPUs as at least one shard per GPU.  The control is config 3 of
bench.py (3.1 Gbases + 5 M variants, ~3.5 Gbases: one shard per GPU).  Both run 100 guides at k = 6 on 1 GPU and on every
visible GPU; per leg one untimed run, then the median of --reps timed runs (context creation, upload from host memory,
scan, device-side resolution, merge).  Prints ONE JSON line (also written to --out) with the GPU name and power limit read
in the same run.
usage: tools/large_text_bench.py [--reps N] [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import varscot_b200 as V                      # noqa: E402
from varscot_b200 import synth                # noqa: E402

N_GUIDES, K = 100, 6


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    rows = [r.split(", ") for r in q.stdout.strip().splitlines()] if q.returncode == 0 else []
    return {"gpu": rows[0][0] if rows else None, "power_limit": rows[0][1] if rows else None, "visible_gpus": V.device_count()}


def leg(text, guides, devices, reps):
    V.map_records(text, guides, K, devices=devices, threads=16)          # untimed: module load, first contexts
    walls, n_rec = [], 0
    for _ in range(reps):
        t = time.perf_counter()
        rec, _, st = V.map_records(text, guides, K, devices=devices, threads=16)
        walls.append(time.perf_counter() - t)
        n_rec = len(rec)
    walls.sort()
    wall = walls[len(walls) // 2]
    n_words = text.n_words
    beyond = n_words * 32 > (1 << 32)
    shards = max(len(devices), -(-n_words // ((1 << 27) - 256))) if beyond else len(devices)     # as vs::shard_plan
    shards = -(-shards // len(devices)) * len(devices)
    return {"gpus": len(devices), "shards": shards, "wall_s": round(wall, 3), "walls_s": [round(w, 3) for w in walls],
            "guide_gbp_per_s": round(N_GUIDES * text.n_bases / 1e9 / wall, 1), "records": n_rec, "device_total_ms": round(st.total_ms, 1)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if V.device_count() < 1:
        sys.exit("large_text_bench: no CUDA device visible")
    guides = synth.synth_guides(13, N_GUIDES)
    out = {"metric": "vs_map_records wall time, 100 guides, k = 6", **gpu_info()}
    all_dev = list(range(V.device_count()))
    for name, gbases, nvar in (("large_5.5G_genome_5M_variants", 5_500_000_000, 5_000_000), ("control_cfg3_3.1G_genome_5M_variants", 3_100_000_000, 5_000_000)):
        t = time.perf_counter()
        text = synth.build_workload(gbases, nvar)
        res = {"n_bases": int(text.n_bases), "n_contigs": int(text.n_contigs), "gen_s": round(time.perf_counter() - t, 1),
               "1gpu": leg(text, guides, [0], args.reps)}
        if len(all_dev) > 1:
            res["all_gpus"] = leg(text, guides, all_dev, args.reps)
        out[name] = res
        del text
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
