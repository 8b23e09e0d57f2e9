#!/bin/bash
# Build libasyncrl_b200.so in-tree for sm_100a.  Usage: csrc/build.sh [extra nvcc flags]
set -euo pipefail
cd "$(dirname "$0")"
OUT=../libasyncrl_b200.so
NVCC=${NVCC:-/usr/local/cuda/bin/nvcc}
SRCS="api.cu preprocess.cu convs_tc.cu reduce.cu fc.cu heads.cu update.cu comm.cu nature.cu lstm.cu"
FLAGS="-gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xcompiler -fPIC -Xcompiler -fvisibility=hidden"
mkdir -p build
pids=()
for s in $SRCS; do
  $NVCC $FLAGS "$@" -c "$s" -o "build/${s%.cu}.o" &
  pids+=($!)
done
for p in "${pids[@]}"; do wait "$p"; done
$NVCC -shared -o "$OUT" $(for s in $SRCS; do echo "build/${s%.cu}.o"; done) -lcudart -ldl
echo "built $(readlink -f $OUT)"
