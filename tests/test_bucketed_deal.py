"""The deal of a batch's guide segments to the warps of k_score_bucketed (vs::bk_deal), run on the HOST by tests/cpu_deal_units.cpp:
every segment is dealt exactly once in the shape the kernel walks, and the most loaded warp stays within the longest-first bound
(1.25 x a lower bound of the best deal) over class counts of 1..32768 guides and K = 0..8.  Dealt round robin, 100 guides break
that bound: the warp that draws a bucket's one 32-guide segment also draws its share of the 4-guide ones."""
import os
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_deal_covers_every_segment_once_within_the_longest_first_bound(tmp_path):
    exe = str(tmp_path / "deal_units")
    r = subprocess.run(["g++", "-O1", "-std=c++20", "-pthread", "-Wno-unknown-pragmas", "-o", exe, os.path.join(ROOT, "tests", "cpu_deal_units.cpp")],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "deal units ok" in r.stdout, r.stdout + r.stderr[-4000:]
