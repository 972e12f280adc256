#!/bin/bash
# Builds the engine of another revision next to the in-tree one, for A/B timing on one GPU box:
#     tools/build_ab.sh <git-rev> [name] [extra nvcc flags, e.g. -DH2SHA_DEBUG_TIMING=2]   ->  tools/ab/libh2sha_<name>.so   (default name: base)
# <git-rev> may be WORK for the working tree as it is.  engine.cu is linked with every *.cc source that revision has.
# then e.g.  TUNE_SUSTAIN=1 TUNE_LIB=tools/ab/libh2sha_base.so python tools/tune.py cfg2 parts=3   (tools/ab.sh interleaves A and B).
# tools/ab/ is scratch: delete it before committing a round (the .so files are git-ignored but would ship to the GPU box).
set -euo pipefail
rev=${1:?usage: build_ab.sh <git-rev> [name] [nvcc flags]}; name=${2:-base}; extra=${3:-}
root="$(cd "$(dirname "$0")/.." && pwd)"
tmp=$(mktemp -d)
mkdir -p "$tmp/halo2-dynamic-sha256_b200/csrc" "$tmp/include" "$root/tools/ab"
if [ "$rev" = WORK ]; then
  cp -r "$root/halo2-dynamic-sha256_b200/csrc/." "$tmp/halo2-dynamic-sha256_b200/csrc/"; cp -r "$root/include/." "$tmp/include/"
else
  for f in $(git -C "$root" ls-tree -r --name-only "$rev" halo2-dynamic-sha256_b200/csrc include); do
    mkdir -p "$tmp/$(dirname "$f")"; git -C "$root" show "$rev:$f" > "$tmp/$f"
  done
fi
/usr/local/cuda/bin/nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -shared -Xcompiler -fPIC -cudart shared -ldl $extra \
  -o "$root/tools/ab/libh2sha_$name.so" "$tmp/halo2-dynamic-sha256_b200/csrc/engine.cu" "$tmp"/halo2-dynamic-sha256_b200/csrc/*.cc
rm -rf "$tmp"
echo "$root/tools/ab/libh2sha_$name.so"
