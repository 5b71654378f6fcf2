#!/bin/bash
# Builds libekfslam.so in-tree for sm_100a.  Usage: build.sh [extra nvcc flags]
set -e
HERE="$(cd "$(dirname "${BASH_SOURCE[0]}")" && pwd)"
OUT="$HERE/../libekfslam.so"
NVCC="${NVCC:-/usr/local/cuda/bin/nvcc}"
FLAGS="-gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xcompiler -fPIC -fmad=true"
mkdir -p "$HERE/build"
pids=()
for f in k_model k_map k_ransac k_update k_chol_big k_downdate k_eval k_cam_update abi; do
  ( "$NVCC" $FLAGS "$@" -c "$HERE/$f.cu" -o "$HERE/build/$f.o" ) &
  pids+=($!)
done
for p in "${pids[@]}"; do wait "$p"; done
"$NVCC" -gencode arch=compute_100a,code=sm_100a -shared -o "$OUT" "$HERE"/build/k_model.o "$HERE"/build/k_map.o "$HERE"/build/k_ransac.o "$HERE"/build/k_update.o "$HERE"/build/k_chol_big.o "$HERE"/build/k_downdate.o "$HERE"/build/k_eval.o "$HERE"/build/k_cam_update.o "$HERE"/build/abi.o -lcudart
echo "built $OUT"
