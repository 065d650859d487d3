#!/bin/bash
# Builds libseedrl_b200.so (sm_100a only) in-tree.  Usage: csrc/build.sh [extra nvcc flags]
set -e
cd "$(dirname "$0")"
NVCC=${NVCC:-/usr/local/cuda/bin/nvcc}
OUT=../libseedrl_b200.so
SRCS="capi.cu vtrace_kernels.cu r2d2_kernels.cu optim_kernels.cu conv_kernels.cu conv_tc_kernels.cu conv_planes.cu conv_first.cu convgen_kernels.cu gemm_kernels.cu gemm_tc_kernels.cu lstm_tiled.cu net_common.cu net.cu r2d2_net.cu store_kernels.cu batcher.cc"
mkdir -p build
OBJS=""
pids=""
for f in $SRCS; do
  o=build/${f%.*}.o
  OBJS="$OBJS $o"
  if [ ! -f "$o" ] || [ "$f" -nt "$o" ] || [ common.cuh -nt "$o" ] || [ kernels.h -nt "$o" ] || [ tc_common.cuh -nt "$o" ] || [ r2d2_thread.inl -nt "$o" ] || [ ../../include/seedrl_b200.h -nt "$o" ]; then
    $NVCC -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xcompiler -fPIC \
      -x cu -c "$f" -o "$o" "$@" &
    pids="$pids $!"
  fi
done
for p in $pids; do wait $p; done
$NVCC -gencode arch=compute_100a,code=sm_100a -shared -o $OUT $OBJS -lpthread
echo "built $(readlink -f $OUT)"
