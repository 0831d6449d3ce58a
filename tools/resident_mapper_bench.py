#!/usr/bin/env python
"""Wall times of the resident mapper (varscot_b200.Mapper) against vs_map_records on one GPU (run on the GPU box).

Texts (synthetic, fixed seeds, synth_core): config 3 of bench.py (3.1 Gbase genome + 5 M variants, ~3.5 Gbases: one shard)
and a 7.1 Gbase genome + 5 M variants (~7.5 Gbases: two shards, both resident on the one device).  Guide sets: 100 guides at
k = 6, and 1000 guides at k = 6 with -P AG.  For every text and guide set, with a host clock around each call (every call
ends in a device synchronise and the host merge):
  * map_records: shard, upload, extract, score, resolve, merge, release — cold on every call (one untimed call first);
  * Mapper create (upload of every shard), the first map (extraction), the second (bucketed build where the library's policy
    builds it), and the median of 5 later maps (steady state).
The records of every Mapper call are compared byte for byte with those of map_records.  Prints ONE JSON line (also written
to --out) with the GPU name, power limit and max SM clock read in the same run.
usage: tools/resident_mapper_bench.py [--out FILE] [--threads T]"""
import argparse
import json
import subprocess
import sys
import os
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import varscot_b200 as V                      # noqa: E402
from varscot_b200 import synth                # noqa: E402

TEXTS = (("cfg3_3.1G_genome_5M_variants", 3_100_000_000, 5_000_000), ("7.1G_genome_5M_variants", 7_100_000_000, 5_000_000))
GUIDE_SETS = (("100_guides_k6", 13, 100, 6, None), ("1000_guides_k6_PAG", 14, 1000, 6, "AG"))
LATER_MAPS = 5


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    rows = [r.split(", ") for r in q.stdout.strip().splitlines()] if q.returncode == 0 else []
    return {"gpu": rows[0][0] if rows else None, "power_limit": rows[0][1] if rows else None,
            "clocks_max_sm": rows[0][2] if rows else None, "visible_gpus": V.device_count()}


def timed(fn):
    t = time.perf_counter()
    out = fn()
    return out, round(time.perf_counter() - t, 4)


def leg(text, guides, k, pam, threads):
    (want, _, st_cold), cold_s = timed(lambda: V.map_records(text, guides, k, pam=pam, devices=[0], threads=threads))
    res = {"records": len(want), "map_records_s": cold_s, "map_records_device_total_ms": round(st_cold.total_ms, 1)}
    m, res["create_s"] = timed(lambda: V.Mapper(text, devices=[0]))
    try:
        res["n_shards"], res["planned_bytes"] = m.n_shards, m.planned_bytes
        calls, same = [], True
        for _ in range(2 + LATER_MAPS):
            (rec, _, st), s = timed(lambda: m.map(guides, k, pam=pam, threads=threads))
            same = same and rec.tobytes() == want.tobytes()
            calls.append({"wall_s": s, "index_reused": st.index_reused, "index_build_ms": round(st.index_build_ms, 2),
                          "device_total_ms": round(st.total_ms, 2), "score_ms": round(st.score_ms, 2), "resolve_ms": round(st.resolve_ms, 2)})
        later = sorted(c["wall_s"] for c in calls[2:])
        res.update({"first_map": calls[0], "second_map": calls[1], "later_maps": calls[2:], "steady_map_s": later[len(later) // 2],
                    "device_bytes": m.device_bytes, "records_identical_to_map_records": same})
    finally:
        m.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="")
    ap.add_argument("--threads", type=int, default=16)
    args = ap.parse_args()
    if V.device_count() < 1:
        sys.exit("resident_mapper_bench: no CUDA device visible")
    out = {"metric": "wall time per call, map_records (cold) vs the resident Mapper, one GPU", **gpu_info()}
    ok = True
    for name, gbases, nvar in TEXTS:
        t = time.perf_counter()
        text = synth.build_workload(gbases, nvar)
        res = {"n_bases": int(text.n_bases), "n_contigs": int(text.n_contigs), "gen_s": round(time.perf_counter() - t, 1)}
        V.map_records(text, synth.synth_guides(13, 8), 4, devices=[0])          # untimed: module load, first contexts
        for gname, seed, n, k, pam in GUIDE_SETS:
            r = leg(text, synth.synth_guides(seed, n), k, pam, args.threads)
            ok = ok and r["records_identical_to_map_records"]
            res[gname] = r
        out[name] = res
        del text
    out["all_mapper_records_identical"] = ok
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
