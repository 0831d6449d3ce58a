#!/bin/bash
# oracle/ref_hook/build_ref.sh <VARSCOT checkout> — TEST INFRASTRUCTURE.  Derives two artefacts from a checkout of the upstream
# VARSCOT repository, outputs ONLY into oracle/_ref/ (git-ignored):
#
#  1. oracle/_ref/VARSCOT           the reference's own driver script (VARSCOT_pipeline/VARSCOT) with its two stray
#                                   `then` lines removed (`else` followed by `then` at :297-298 and :312-313 makes bash
#                                   reject the shipped file: `bash -n` fails).  Nothing else is touched, so a test that
#                                   runs it against our six executables is a test of the drop-in boundary at driver level.
#  2. oracle/_ref/bidir_mapping,    the TRUE reference read mapper, built with the reference's own CMake project
#     oracle/_ref/bidir_index       (VARSCOT_pipeline/read_mapping/CMakeLists.txt) — ONLY when a SeqAn 2.4.0rc2 checkout
#                                   exists at $SEQAN_DIR or <reference>/VARSCOT_pipeline/lib/seqan (the reference clones it
#                                   at docker-build time, Dockerfile:41; without it this step reports "unbuildable"
#                                   and parity stays unpinned).  The day it is supplied,
#                                   tools/diff_against_ref.sh diffs the oracle and the CUDA mapper against it.
set -u
HERE="$(cd "$(dirname "$0")" && pwd)"
REF="${1:?usage: build_ref.sh <checkout of the upstream VARSCOT repository>}"
OUT="$HERE/../_ref"
[ -d "$REF/VARSCOT_pipeline" ] || { echo "build_ref: no reference tree at $REF (nothing to do)"; exit 0; }
mkdir -p "$OUT"
# 1. driver script: drop a `then` line that directly follows an `else` line
awk '{ if (prev_else && $0 ~ /^[[:space:]]*then[[:space:]]*$/) { prev_else = 0; next } prev_else = ($0 ~ /^[[:space:]]*else[[:space:]]*$/); print }' \
    "$REF/VARSCOT_pipeline/VARSCOT" > "$OUT/VARSCOT" && chmod +x "$OUT/VARSCOT"
if bash -n "$OUT/VARSCOT"; then echo "build_ref: oracle/_ref/VARSCOT parses ($(diff <(cat "$REF/VARSCOT_pipeline/VARSCOT") "$OUT/VARSCOT" | grep -c '^<') lines removed)"
else echo "build_ref: the patched driver still does not parse"; rm -f "$OUT/VARSCOT"; fi
# 2. the true mapper, if SeqAn is there
SEQAN="${SEQAN_DIR:-$REF/VARSCOT_pipeline/lib/seqan}"
if [ -f "$SEQAN/include/seqan/index.h" ] && command -v cmake >/dev/null; then
    B="$(mktemp -d)"
    # the project expects ../lib/seqan next to read_mapping/: build from a scratch copy of the two directories' layout (links only)
    mkdir -p "$B/src/lib" && ln -s "$REF/VARSCOT_pipeline/read_mapping" "$B/src/read_mapping" && ln -s "$SEQAN" "$B/src/lib/seqan"
    if cmake -S "$B/src/read_mapping" -B "$B/build" -DCMAKE_BUILD_TYPE=Release >/dev/null && cmake --build "$B/build" -j >/dev/null; then
        cp "$B/build/bidir_mapping" "$B/build/bidir_index" "$OUT/" && echo "build_ref: built oracle/_ref/bidir_mapping + bidir_index from the reference sources"
    else echo "build_ref: SeqAn found but the reference build failed"; fi
    rm -rf "$B"
else
    echo "build_ref: SeqAn 2.4.0rc2 not found at $SEQAN: the reference mapper is unbuildable here (parity unpinned)"
fi
