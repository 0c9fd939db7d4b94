#!/usr/bin/env bash
# Debug build with per-tile phase timelines in the tile GEMM: gpr.jl_b200/libgprb200_tl.so (use via GPRB200_LIB=...)
set -euo pipefail
cd "$(dirname "$0")"
NVCC=${NVCC:-/usr/local/cuda/bin/nvcc}
FLAGS=(-gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xcompiler -fPIC -DGPRB_TIMELINE)
mkdir -p build/tl
for f in api tilegemm covgrad factor predict postcov loo predgrad lbfgs comm; do "$NVCC" "${FLAGS[@]}" -c "$f.cu" -o "build/tl/$f.o" 2>/dev/null & done
wait
"$NVCC" -shared -o ../libgprb200_tl.so build/tl/*.o -lcudart -ldl
echo "built ../libgprb200_tl.so"
