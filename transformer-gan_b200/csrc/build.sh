#!/bin/bash
# Builds libtgan_b200.so (sm_100a only) next to the Python package.  Usage: csrc/build.sh [-j N]
set -e
HERE="$(cd "$(dirname "${BASH_SOURCE[0]}")" && pwd)"
OUT="$HERE/../tgan_b200"
OBJ="$HERE/build"
mkdir -p "$OBJ" "$OUT"
NVCC="${NVCC:-/usr/local/cuda/bin/nvcc}"
FLAGS="-gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xcompiler -fPIC -Xptxas -v"
pids=()
for f in rowops gemm_simt gemm_tc relattn relattn_simt relattn_decode bert_ops bert_attn_mma sampling ring_scatter batching nccl_bucket relattn_tc relattn_fwd_tc; do
  if [ ! -f "$OBJ/$f.o" ] || [ "$HERE/$f.cu" -nt "$OBJ/$f.o" ] || [ "$HERE/common.cuh" -nt "$OBJ/$f.o" ] || \
     [ "$HERE/tc_common.cuh" -nt "$OBJ/$f.o" ] || [ "$HERE/../../include/tgan_b200.h" -nt "$OBJ/$f.o" ]; then
    ( $NVCC $FLAGS -c "$HERE/$f.cu" -o "$OBJ/$f.o" > "$OBJ/$f.log" 2>&1 || { cat "$OBJ/$f.log"; exit 1; } ) &
    pids+=($!)
  fi
done
for p in "${pids[@]}"; do wait $p; done
$NVCC -shared -o "$OUT/libtgan_b200.so" "$OBJ"/rowops.o "$OBJ"/gemm_simt.o "$OBJ"/gemm_tc.o "$OBJ"/relattn.o \
      "$OBJ"/relattn_simt.o "$OBJ"/relattn_decode.o "$OBJ"/bert_ops.o "$OBJ"/bert_attn_mma.o "$OBJ"/sampling.o "$OBJ"/ring_scatter.o "$OBJ"/batching.o "$OBJ"/nccl_bucket.o "$OBJ"/relattn_tc.o "$OBJ"/relattn_fwd_tc.o -lcudart -ldl
echo "built $OUT/libtgan_b200.so"
