#!/bin/bash
# Builds ipdm-pytorch_b200/libipdm_b200.so for sm_100a (cross-compiles without a GPU).
set -e
cd "$(dirname "$0")"
NVCC=${NVCC:-/usr/local/cuda/bin/nvcc}
OUT=../libipdm_b200.so
FLAGS="-gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xcompiler -fPIC -Xcompiler -Wall -Xptxas -v --expt-relaxed-constexpr"
mkdir -p _obj
pids=()
for f in api fbp project sart sampler unet_kernels conv_tc conv_thin attention unet engine metrics; do
  if [ ! -f _obj/$f.o ] || [ $f.cu -nt _obj/$f.o ] || [ common.cuh -nt _obj/$f.o ] || [ tc.cuh -nt _obj/$f.o ] || [ unet_ops.cuh -nt _obj/$f.o ] || [ fbp_plan.cuh -nt _obj/$f.o ] || [ ../../include/ipdm_b200.h -nt _obj/$f.o ]; then
    ( $NVCC $FLAGS -c $f.cu -o _obj/$f.o > _obj/$f.log 2>&1 || { cat _obj/$f.log; exit 1; } ) &
    pids+=($!)
  fi
done
for p in "${pids[@]}"; do wait $p; done
$NVCC -shared -o $OUT _obj/*.o -gencode arch=compute_100a,code=sm_100a
echo "built $(realpath $OUT)"
