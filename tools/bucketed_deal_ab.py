#!/usr/bin/env python
"""A/B of the resident bucketed scan: this tree's library against a second build (usually the parent commit), in one process
tree on one GPU, runs alternating so that drift of the card or the host hits both builds alike.

usage: tools/bucketed_deal_ab.py OTHER_TREE [--runs 3] [--extra-configs 4 2] [--out FILE]
  OTHER_TREE  a checkout of the other version (e.g. `git archive <parent> | tar -x -C OTHER_TREE`); its library is built there
              with its own Makefile unless OTHER_TREE/varscot_b200/libvarscot_scan.so exists.  This tree's library must be built.

Per run: `bench.py --config 3 --no-cpu --no-dense --no-cli --dump-outputs D` with VARSCOT_LIB naming the build, A B A B ...;
then each extra config once per build (`--no-cpu --no-dense --no-cli --no-target --no-e2e`, also dumped).  Every dump of one
build is compared array for array with the dump of the other build at the same config (the first run's for config 3).  The
JSON written to --out (and printed) holds the per-run bench lines reduced to their timings, the spread of each build, the
ratios of the medians, the output comparison, and the card: name, power limit, SM clocks (nvidia-smi, same call)."""
import argparse
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join("varscot_b200", "libvarscot_scan.so")


def card():
    q = "name,power.limit,power.max_limit,clocks.sm,clocks.max.sm,driver_version"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                             timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        return {"error": str(e)}
    return dict(zip(q.split(","), [x.strip() for x in out.split(",")]))


def bench(lib, config, dump, extra):
    env = dict(os.environ, VARSCOT_LIB=lib)
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--config", str(config), "--no-cpu", "--no-dense", "--no-cli",
           "--dump-outputs", dump, *extra]
    r = subprocess.run(cmd, capture_output=True, text=True, env=env, cwd=ROOT)
    lines = [x for x in r.stdout.splitlines() if x.startswith("{")]
    if r.returncode != 0 or not lines:
        raise RuntimeError(f"bench failed ({r.returncode}): {' '.join(cmd)}\n{r.stdout[-3000:]}\n{r.stderr[-3000:]}")
    return json.loads(lines[-1])


def reduce(line):
    """the timings and parity fields of a bench line"""
    ph = line.get("phase_ms_rank0") or {}
    out = {"ms_per_step": line.get("ms_per_step"), "score_ms": ph.get("score"), "value": line.get("value"),
           "index_lists_identical": line.get("index_lists_identical"), "hits_per_step": line.get("hits_per_step"),
           "sm_mhz": (line.get("clocks") or {}).get("sm_mhz"), "clock_reasons": (line.get("clocks") or {}).get("reasons")}
    t = line.get("target_cfg4")
    if isinstance(t, dict) and "ms_per_step" in t:
        out["cfg4_ms_per_step"] = t["ms_per_step"]
        out["cfg4_score_ms"] = (t.get("phase_ms_rank0") or {}).get("score")
        out["cfg4_index_lists_identical"] = t.get("index_lists_identical")
    return out


def same_arrays(d1, d2):
    import numpy as np
    n1, n2 = sorted(os.listdir(d1)), sorted(os.listdir(d2))
    if n1 != n2 or not n1:
        return {"identical": False, "why": f"files differ: {n1} vs {n2}"}
    diff = [n for n in n1 if not np.array_equal(np.load(os.path.join(d1, n)), np.load(os.path.join(d2, n)))]
    return {"identical": not diff, "arrays": len(n1), "differing": diff}


def spread(xs):
    xs = [x for x in xs if x is not None]
    return {"median": statistics.median(xs), "min": min(xs), "max": max(xs), "runs": xs} if xs else None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("other_tree")
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--extra-configs", type=int, nargs="*", default=[4, 2])
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    new_lib = os.path.join(ROOT, LIB)
    old_lib = os.path.join(os.path.abspath(args.other_tree), LIB)
    if not os.path.exists(new_lib):
        sys.exit(f"{new_lib} is missing: build this tree first")
    if not os.path.exists(old_lib):
        r = subprocess.run(["make", "-C", args.other_tree, LIB], capture_output=True, text=True)
        if r.returncode != 0:
            sys.exit("building the other tree failed:\n" + r.stdout[-2000:] + r.stderr[-2000:])
    builds = {"new": new_lib, "old": old_lib}
    tmp = tempfile.mkdtemp(prefix="vs_ab_")
    res = {"card_before": card(), "builds": {"new": ROOT, "old": os.path.abspath(args.other_tree)},
           "command": "bench.py --gpus 1 --config 3 --no-cpu --no-dense --no-cli", "runs": {"new": [], "old": []}}
    try:
        for i in range(args.runs):
            for name in ("new", "old") if i % 2 == 0 else ("old", "new"):
                d = os.path.join(tmp, f"c3_{name}_{i}")
                res["runs"][name].append(reduce(bench(builds[name], 3, d, [])))
                print(name, i, json.dumps(res["runs"][name][-1]), flush=True)
        res["outputs_cfg3"] = [same_arrays(os.path.join(tmp, f"c3_new_{i}"), os.path.join(tmp, f"c3_old_{i}")) for i in range(args.runs)]
        res["summary_cfg3"] = {}
        for key in ("score_ms", "ms_per_step", "cfg4_ms_per_step", "cfg4_score_ms"):
            s = {name: spread([r.get(key) for r in res["runs"][name]]) for name in ("new", "old")}
            if s["new"] and s["old"]:
                s["old_over_new"] = s["old"]["median"] / s["new"]["median"]
            res["summary_cfg3"][key] = s
        for cfg in args.extra_configs:
            lines = {}
            for name in ("new", "old"):
                lines[name] = reduce(bench(builds[name], cfg, os.path.join(tmp, f"c{cfg}_{name}"), ["--no-target", "--no-e2e"]))
                print(name, f"cfg{cfg}", json.dumps(lines[name]), flush=True)
            lines["outputs"] = same_arrays(os.path.join(tmp, f"c{cfg}_new"), os.path.join(tmp, f"c{cfg}_old"))
            lines["old_over_new_ms_per_step"] = lines["old"]["ms_per_step"] / lines["new"]["ms_per_step"]
            res[f"config{cfg}"] = lines
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    res["card_after"] = card()
    txt = json.dumps(res)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(txt + "\n")
    print(txt)


if __name__ == "__main__":
    main()
