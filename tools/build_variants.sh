#!/bin/bash
# Build liboptb from named commits into build_variants/liboptb_<name>.so (git-ignored via *.so) for
# tools/variant_bench.py, e.g. the parent of a change and the change itself:
#   tools/build_variants.sh parent HEAD~1 new HEAD
# Each commit's sources are exported with `git archive`, so the working tree is not touched.
set -e
ROOT="$(cd "$(dirname "$0")/.." && pwd)"
OUT="$ROOT/build_variants"
TMP="$(mktemp -d)"
trap 'rm -rf "$TMP"' EXIT
mkdir -p "$OUT"
pids=()
while [ $# -ge 2 ]; do
  name="$1"; commit="$2"; shift 2
  mkdir -p "$TMP/$name"
  git -C "$ROOT" archive "$commit" optable_b200/csrc include | tar -x -C "$TMP/$name"
  ( cd "$TMP/$name/optable_b200/csrc" \
      && nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xcompiler -fPIC -shared -ldl \
           -o "$OUT/liboptb_$name.so" optb.cu \
      && echo "built $name ($commit)" ) &
  pids+=($!)
  if [ ${#pids[@]} -ge 4 ]; then wait "${pids[0]}"; pids=("${pids[@]:1}"); fi
done
for p in "${pids[@]}"; do wait "$p"; done
