"""Generates the committed golden fixtures under tests/golden/:  python tests/golden/make_golden.py [<VARSCOT checkout>]

* ref_guides.fa : the 16 real guides the reference ships as inputs for this path
  (workflow/guideseq-data/guideseqOntargets.fasta, workflow/siteseq-data/siteseqOntargets.fasta) —
  input data only; the reference holds NO expected outputs for bidir_mapping (its one golden SAM is a
  git-LFS pointer), so parity stays "unpinned".  Rewritten only when a checkout of upstream VARSCOT is given.
* case_*.json   : small seeded cases with the ORACLE's records and SAM text; they pin the oracle against
  accidental change and give the GPU tests an oracle-independent file to compare with.
"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import oracle as O          # noqa: E402
from tests.util import make_case        # noqa: E402


def ref_guides(workflow):
    out = []
    for f in ("guideseq-data/guideseqOntargets.fasta", "siteseq-data/siteseqOntargets.fasta"):
        out.append(open(os.path.join(workflow, f)).read())
    open(os.path.join(HERE, "ref_guides.fa"), "w").write("".join(out))


def dump_case(name, case, md_style=O.MD_SEQAN):
    codes = O.text_codes(case.ascii)
    r = O.map_guides(codes, case.offsets, case.guides, case.k, pam=case.pam, md_style=md_style)
    assert O.map_guides(codes, case.offsets, case.guides, case.k, pam=case.pam, mode=O.MODE_LITERAL, md_style=md_style).rows() == r.rows()
    json.dump({"ascii": case.ascii.decode(), "offsets": [int(x) for x in case.offsets], "guides": case.guide_strs, "k": case.k,
               "pam": case.pam, "names": case.names,
               "rows": [list(x) for x in r.rows()]}, open(os.path.join(HERE, name + ".json"), "w"))
    print(name, len(r), "records")


if __name__ == "__main__":
    if len(sys.argv) > 1:
        ref_guides(os.path.join(sys.argv[1], "workflow"))
    dump_case("case_k4", make_case(seed=1001, contig_lens=[6000, 45, 45, 23, 0, 22, 3000], n_guides=4, k=4))
    dump_case("case_k6_pamAG", make_case(seed=1002, contig_lens=[8000, 45, 2000], n_guides=5, k=6, pam="AG"))
    dump_case("case_k8", make_case(seed=1003, contig_lens=[5000, 46, 47, 1000], n_guides=3, k=8))
    dump_case("case_k0", make_case(seed=1004, contig_lens=[4000, 4000], n_guides=6, k=0))
    # the reference's real guides on a random text with planted sites
    gs = [l.strip() for l in open(os.path.join(HERE, "ref_guides.fa")) if not l.startswith(">")]
    case = make_case(seed=1005, contig_lens=[20000, 45, 45, 5000], n_guides=len(gs), k=5)
    rng = np.random.default_rng(77)
    asc = np.frombuffer(case.ascii, dtype=np.uint8).copy()
    case.guides = O.guide_codes(gs); case.guide_strs = gs
    lut = np.frombuffer(b"ACGT", dtype=np.uint8)
    for i, g in enumerate(case.guides):
        for j in range(4):
            w = g.copy()
            idx = rng.choice(23, j + 1, replace=False); w[idx] = (w[idx] + 1) % 4
            if j % 2:
                w = (3 - w[::-1]).astype(np.uint8)
            p = int(rng.integers(0, 20000 - 23))
            asc[p:p + 23] = lut[w]
    case.ascii = bytes(asc)
    dump_case("case_refguides_k5", case)
