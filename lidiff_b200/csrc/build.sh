#!/usr/bin/env bash
# Builds lidiff_b200/_C/liblidiff_b200.so for sm_100a (cross-compiles without a GPU).
set -euo pipefail
here="$(cd "$(dirname "$0")" && pwd)"
out="$here/../_C"
mkdir -p "$out"
NVCC=${NVCC:-/usr/local/cuda/bin/nvcc}
FLAGS=(-gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xcompiler -fPIC -Xptxas -v)
objs=()
for f in coords spconv_ffma spconv_tc spconv_tc2 spconv_tc3 spconv_tc4 spconv_tc5 spconv_scatter dense metrics api; do
  src="$here/$f.cu"; obj="$out/$f.o"
  if [ ! -f "$obj" ] || [ "$src" -nt "$obj" ] || [ "$here/common.cuh" -nt "$obj" ] || [ "$here/tc_common.cuh" -nt "$obj" ] || [ "$here/../../include/lidiff_b200.h" -nt "$obj" ]; then
    "$NVCC" "${FLAGS[@]}" -c "$src" -o "$obj" 2> "$out/$f.ptxas.log" || { cat "$out/$f.ptxas.log"; exit 1; }
  fi
  objs+=("$obj")
done
"$NVCC" -shared -gencode arch=compute_100a,code=sm_100a -o "$out/liblidiff_b200.so" "${objs[@]}" -lcudart
echo "built $out/liblidiff_b200.so"
