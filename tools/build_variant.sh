#!/bin/bash
# Build the engine library of another git revision into <out.so> for same-box A/B timing:
#   tools/build_variant.sh <git-rev> glom_pytorch_b200/libglom_b200_A.so
#   GLOM_B200_LIB=glom_pytorch_b200/libglom_b200_A.so python tools/diag.py timing
# The revision is compiled by its own build.py, so the source list always matches that revision.
set -e
rev=$1; out=$(realpath -m "$2"); tmp=$(mktemp -d)
trap 'rm -rf "$tmp"' EXIT
git archive "$rev" glom_pytorch_b200 include | tar -x -C "$tmp"
mkdir "$tmp/out"
( cd "$tmp" && python -c "from glom_pytorch_b200.build import build_library; build_library(out_dir='out')" )
cp "$tmp/out/libglom_b200.so" "$out"
echo "$out"
