#!/usr/bin/env python
"""Streamed records (Mapper.map_stream, bidir_mapping's streamed SAM) against the one-shot calls, on one GPU (run on the GPU box).

Text: config 3 of bench.py (3.1 Gbase genome + 5 M variants, ~3.5 Gbases, fixed seeds), built once and saved as a packed-text
cache in a temporary directory; every leg runs in a child process that loads it, so that each reports its own peak RSS and
imports the package of the build it measures (this tree, or --parent-root: a checkout of the parent commit with its library
built).  Peak RSS is the child's VmHWM (a child inherits its parent's ru_maxrss across exec, so the text is built in a child
too).  Host clocks are taken around calls that end in a device synchronise.
  existing  this build and its parent, alternated twice: the steady Mapper.map (median of 5 after two warm
            calls) at 100 guides k <= 6 and at 1000 guides k <= 6 -P AG, and a cold map_records at 100 guides k <= 6
  dense     1000 guides, k <= 8: Mapper.map against map_stream with a counting sink, without and with windows
  exe       bidir_mapping -M 8 -T 16 with 100 guides on the cache, this build and its parent alternated: wall time, the
            VARSCOT_VERBOSE phases, max RSS and the SAM's sha256 (must match)
  config5   10 000 guides, k <= 8 (~1.9e9 records) through Mapper.map_stream with a per-guide counting sink; the peak RSS
            against the documented bound; the per-guide totals against a plain vs_scan_resolved sink's per-guide count
Prints ONE JSON line (also written to --out) with the GPU name, power limit and max SM clock read in the same run.
usage: tools/record_stream_bench.py --parent-root DIR [--out FILE] [--skip LEG ...] [--existing-reps N]"""
import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GENOME, VARIANTS = 3_100_000_000, 5_000_000
RPD = 32 << 20                                   # the library's default records per delivery


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    rows = [r.split(", ") for r in q.stdout.strip().splitlines()] if q.returncode == 0 else []
    return {"gpu": rows[0][0] if rows else None, "power_limit": rows[0][1] if rows else None, "clocks_max_sm": rows[0][2] if rows else None}


def timed(fn):
    t = time.perf_counter()
    out = fn()
    return out, round(time.perf_counter() - t, 4)


def peak_rss_bytes():
    with open("/proc/self/status") as f:
        for line in f:
            if line.startswith("VmHWM:"):
                return int(line.split()[1]) * 1024
    return 0


# ---- child legs (this process imports the package of the build under `root`) ----------------------------------------------------
def child(leg, prefix, root):
    sys.path.insert(0, root)
    import numpy as np
    import varscot_b200 as V
    from varscot_b200 import synth
    if leg == "build":                                   # the packed-text cache every other leg loads
        text = synth.build_workload(GENOME, VARIANTS)
        text.save(prefix)
        with open(prefix + ".vsnames", "w") as f:
            f.write("".join(f"seq{i}\n" for i in range(text.n_contigs)))
        with open(prefix + ".fa", "w") as f:
            f.write(">unused\nA\n")                        # ids come from .vsnames
        print("RESULT " + json.dumps({"n_bases": int(text.n_bases), "n_contigs": int(text.n_contigs)}))
        return
    text = V.PackedText.load(prefix)
    base_rss = peak_rss_bytes()
    out = {"text_rss_bytes": base_rss}
    if leg == "existing":
        with V.Mapper(text, devices=[0]) as m:
            for name, seed, n, k, pam in (("100_guides_k6", 13, 100, 6, None), ("1000_guides_k6_PAG", 14, 1000, 6, "AG")):
                g = synth.synth_guides(seed, n)
                walls = []
                for i in range(7):
                    (rec, _, st), s = timed(lambda: m.map(g, k, pam=pam, threads=16))
                    if i >= 2:
                        walls.append(s)
                out[name] = {"steady_map_s": statistics.median(walls), "records": len(rec), "device_total_ms": round(st.total_ms, 2),
                             "sha256": hashlib.sha256(rec.tobytes()).hexdigest()}
        g = synth.synth_guides(13, 100)
        (rec, _, st), s = timed(lambda: V.map_records(text, g, 6, devices=[0], threads=16))
        out["cold_map_records_100_guides_k6"] = {"wall_s": s, "device_total_ms": round(st.total_ms, 1), "sha256": hashlib.sha256(rec.tobytes()).hexdigest()}
    elif leg.startswith("dense_"):
        variant = leg[len("dense_"):]
        g = synth.synth_guides(14, 1000)
        with V.Mapper(text, devices=[0]) as m:
            m.map(synth.synth_guides(13, 8), 8)                          # the index is extracted before the timed call
            if variant == "map":
                (rec, coll, st), s = timed(lambda: m.map(g, 8, threads=16))
                n, digest = len(rec), hashlib.sha256(rec["guide"].tobytes()).hexdigest()
                del rec
            else:
                counts = {"n": 0, "deliveries": 0, "largest": 0}
                h = hashlib.sha256()

                def sink(rec, win, lo, hi):
                    counts["n"] += len(rec)
                    counts["deliveries"] += 1
                    counts["largest"] = max(counts["largest"], len(rec))
                    h.update(rec["guide"].tobytes())
                (coll, st), s = timed(lambda: m.map_stream(g, 8, sink, threads=16, windows=variant == "stream_windows"))
                n, digest = counts["n"], h.hexdigest()
                out.update(deliveries=counts["deliveries"], largest_delivery=counts["largest"])
        out.update(wall_s=s, records=n, device_total_ms=round(st.total_ms, 1), resolve_ms=round(st.resolve_ms, 1), d2h_bytes=st.d2h_bytes,
                   key16_collisions=coll, guide_ids_sha256=digest)
    elif leg == "config5":
        g = synth.synth_guides(15, 10000)
        per_guide = np.zeros(len(g), dtype=np.int64)
        counts = {"deliveries": 0, "largest": 0}

        def sink(rec, win, lo, hi):
            per_guide[lo:hi] += np.bincount(rec["guide"] - lo, minlength=hi - lo)[: hi - lo] if len(rec) else 0
            counts["deliveries"] += 1
            counts["largest"] = max(counts["largest"], len(rec))
        with V.Mapper(text, devices=[0]) as m:
            (coll, st), s = timed(lambda: m.map_stream(g, 8, sink, threads=16))
        peak = peak_rss_bytes()
        # the documented bound: 3 x records_per_delivery x 16 B in flight, plus the context's pinned staging of its largest
        # super-chunk (at most the 64 Mi-hit device buffer + 1/8)
        bound = 3 * RPD * 16 + (64 << 20) * 16 * 9 // 8
        ref = np.zeros(len(g), dtype=np.int64)

        def ref_sink(hits, lo, hi):
            ref[:] += np.bincount(hits["info"] >> 8, minlength=len(g))[: len(g)]
        with V.ScanContext(0) as ctx:
            _, st_ref = ctx.scan_resolved(g, 8, text=text, sink=ref_sink)
        out.update(wall_s=s, records=int(per_guide.sum()), deliveries=counts["deliveries"], largest_delivery=counts["largest"],
                   device_total_ms=round(st.total_ms, 1), key16_collisions=coll, peak_rss_bytes=peak,
                   rss_above_text_bytes=peak - base_rss, documented_bound_bytes=bound, within_bound=peak - base_rss <= bound,
                   reference_hits=int(ref.sum()), per_guide_equal=bool(np.array_equal(per_guide, ref)))
    out["peak_rss_bytes"] = out.get("peak_rss_bytes", peak_rss_bytes())
    print("RESULT " + json.dumps(out))


def run_child(leg, prefix, root):
    env = {k: v for k, v in os.environ.items() if k != "VARSCOT_LIB"}
    r = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", leg, "--prefix", prefix, "--root", root],
                       capture_output=True, text=True, env=env)
    for line in r.stdout.splitlines():
        if line.startswith("RESULT "):
            return json.loads(line[7:])
    return {"error": f"exit {r.returncode}: {r.stderr[-2000:]}"}


def run_exe(prefix, guides_fa, lib_dir, sam):
    exe = os.path.join(ROOT, "build", "read_mapping_build", "bidir_mapping")
    env = dict(os.environ, VARSCOT_VERBOSE="1", LD_LIBRARY_PATH=lib_dir)
    t = time.perf_counter()
    p = subprocess.Popen([exe, "-G", prefix + ".fa", "-I", prefix, "-R", guides_fa, "-M", "8", "-T", "16", "-O", sam],
                         stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, env=env)
    _, _, ru = os.wait4(p.pid, 0)
    wall = time.perf_counter() - t
    err = p.stderr.read()
    h = hashlib.sha256()
    with open(sam, "rb") as f:
        for chunk in iter(lambda: f.read(1 << 24), b""):
            h.update(chunk)
    size = os.path.getsize(sam)
    os.remove(sam)
    return {"wall_s": round(wall, 3), "max_rss_bytes": ru.ru_maxrss * 1024, "sam_bytes": size, "sam_sha256": h.hexdigest(),
            "phases": [l.split(": ", 1)[1] for l in err.splitlines() if "wall:" in l or "upload+scan" in l]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--child", default="")
    ap.add_argument("--prefix", default="")
    ap.add_argument("--root", default=ROOT)
    ap.add_argument("--parent-root", default="")
    ap.add_argument("--out", default="")
    ap.add_argument("--skip", nargs="*", default=[])
    ap.add_argument("--existing-reps", type=int, default=2, help="alternations of the existing leg")
    args = ap.parse_args()
    if args.child:
        return child(args.child, args.prefix, args.root)
    if not args.parent_root or not os.path.exists(os.path.join(args.parent_root, "varscot_b200", "libvarscot_scan.so")):
        sys.exit("record_stream_bench: --parent-root must be a checkout of the parent commit with its library built")
    this, parent = ROOT, os.path.abspath(args.parent_root)
    out = {"metric": "streamed records vs the one-shot calls, config-3 text, one GPU", **gpu_info(),
           "records_per_delivery": RPD}
    with tempfile.TemporaryDirectory() as d:
        prefix = os.path.join(d, "cfg3")
        t = time.perf_counter()
        out["text"] = {**run_child("build", prefix, this), "gen_s": round(time.perf_counter() - t, 1)}
        if "existing" not in args.skip:
            runs = []
            for rep in range(args.existing_reps):
                for name, root in (("parent", parent), ("this", this)):
                    runs.append({"build": name, "rep": rep, **run_child("existing", prefix, root)})
            out["existing"] = runs
        if "dense" not in args.skip:
            out["dense_1000_guides_k8"] = {v: run_child("dense_" + v, prefix, this) for v in ("map", "stream", "stream_windows")}
        if "exe" not in args.skip:
            guides_fa = os.path.join(d, "guides.fa")
            sys.path.insert(0, ROOT)
            from varscot_b200 import synth_core
            g = synth_core.synth_guides(13, 100)
            with open(guides_fa, "w") as f:
                for i, row in enumerate(g):
                    f.write(f">g{i}\n" + "".join("ACGT"[int(b)] for b in row) + "\n")
            runs = []
            for rep in range(2):
                for name, root in (("parent", parent), ("this", this)):
                    runs.append({"build": name, "rep": rep, **run_exe(prefix, guides_fa, os.path.join(root, "varscot_b200"), os.path.join(d, "o.sam"))})
            out["exe_100_guides_M8_T16"] = runs
            out["exe_sam_identical"] = len({r["sam_sha256"] for r in runs}) == 1
        if "config5" not in args.skip:
            out["config5_map_stream"] = run_child("config5", prefix, this)
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
