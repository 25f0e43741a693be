#!/bin/bash
# Builds libb200z.so in-tree for sm_100a (nvcc cross-compiles without a GPU).
set -e
cd "$(dirname "$0")"
# nvcc from $NVCC, else PATH, else the toolkit under $CUDA_HOME (default /usr/local/cuda), which a plain login PATH lacks
NVCC=${NVCC:-$(command -v nvcc || echo "${CUDA_HOME:-/usr/local/cuda}/bin/nvcc")}
FLAGS="-gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xcompiler -fPIC -Xcompiler -Wall -diag-suppress 550"
mkdir -p _build
pids=()
for f in b200z_deflate b200z_inflate b200z_checksum b200z_api b200z_crypto; do
  stale=0
  [ -f _build/$f.o ] || stale=1
  for dep in $f.cu *.cuh ../../include/b200z.h build.sh; do
    [ $stale -eq 0 ] && [ $dep -nt _build/$f.o ] && stale=1
  done
  if [ $stale -eq 1 ]; then
    rm -f _build/$f.o # a failed compile must not leave an older object for the link step
    $NVCC $FLAGS -c $f.cu -o _build/$f.o &
    pids+=($!)
  fi
done
for pid in "${pids[@]}"; do
  wait "$pid" || { echo "build.sh: a compile failed" >&2; exit 1; }
done
$NVCC -gencode arch=compute_100a,code=sm_100a -shared -o ../libb200z.so _build/b200z_deflate.o _build/b200z_inflate.o _build/b200z_checksum.o _build/b200z_api.o _build/b200z_crypto.o
echo built ../libb200z.so
