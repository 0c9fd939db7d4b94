#!/usr/bin/env bash
# Build libgprb200.so (sm_100a only) in-tree: gpr.jl_b200/libgprb200.so
set -euo pipefail
cd "$(dirname "$0")"
OUT=../libgprb200.so
NVCC=${NVCC:-/usr/local/cuda/bin/nvcc}
FLAGS=(-gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xcompiler -fPIC -Xcompiler -O2 -Xptxas -v)
mkdir -p build
pids=()
for f in api tilegemm covgrad factor predict postcov loo predgrad lbfgs comm; do
  [ -f "$f.cu" ] || continue
  if [ ! -f "build/$f.o" ] || [ "$f.cu" -nt "build/$f.o" ] || [ common.cuh -nt "build/$f.o" ] || [ kernels.h -nt "build/$f.o" ] || [ ../../include/gprb200.h -nt "build/$f.o" ]; then
    ( "$NVCC" "${FLAGS[@]}" -c "$f.cu" -o "build/$f.o" > "build/$f.log" 2>&1 || { cat "build/$f.log"; exit 1; } ) &
    pids+=($!)
  fi
done
for p in "${pids[@]:-}"; do [ -n "$p" ] && wait "$p"; done
"$NVCC" -gencode arch=compute_100a,code=sm_100a -shared -o "$OUT" build/*.o -lcudart -ldl
echo "built $OUT"
