#!/bin/bash
# Builds libbsrnn_b200.so in-tree for sm_100a (cross-compiles without a GPU).
set -e
cd "$(dirname "$0")"
SRC=urgent2026_challenge_track1_b200/csrc
OUT=urgent2026_challenge_track1_b200/_C
mkdir -p $OUT
NVCC=${NVCC:-/usr/local/cuda/bin/nvcc}
# no --use_fast_math: the f32-mode kernels call expf/tanhf for parity; approximations are explicit PTX where wanted
FF="-gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xcompiler -fPIC -Xptxas -v $BSRNN_NVCC_FLAGS"
SRCS="api fft norm gemm_f32 lstm_f32 flow pack gemm_tc lstm_tc lstm_fused optim loss bandsplit mix metrics $EXTRA"
pids=""
for f in $SRCS; do
  # rebuild only what changed (sources are independent translation units); compile in parallel
  if [ ! -f $OUT/$f.o ] || [ $SRC/$f.cu -nt $OUT/$f.o ] || [ -n "$(find $SRC -name '*.cuh' -newer $OUT/$f.o)" ] || [ include/bsrnn_b200.h -nt $OUT/$f.o ]; then
    ( $NVCC $FF -c $SRC/$f.cu -o $OUT/$f.o 2> $OUT/$f.ptxas.log || { cat $OUT/$f.ptxas.log; rm -f $OUT/$f.o; exit 1; } ) &
    pids="$pids $!"
  fi
done
for p in $pids; do wait $p || exit 1; done
OBJS=""; for f in $SRCS; do OBJS="$OBJS $OUT/$f.o"; done
$NVCC -shared -o $OUT/libbsrnn_b200.so $OBJS -lcudart
echo built $OUT/libbsrnn_b200.so
