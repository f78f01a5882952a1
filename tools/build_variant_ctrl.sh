#!/bin/bash
# Like build_variant.sh, for experiments on the per-call controller kernel: rebuilds the C ABI file and the ctrl_step TU (kind 1, fp32).
# usage: tools/build_variant_ctrl.sh <tag> "<extra nvcc flags>"  ->  multidronesim_b200/csrc/libmds_<tag>.so
set -e
tag=$1; extra=$2
cd "$(dirname "$0")/../multidronesim_b200/csrc"
make -j8 >/dev/null
mkdir -p build_$tag
FLAGS="-O3 -std=c++17 -lineinfo -use_fast_math -gencode arch=compute_100a,code=sm_100a -Xcompiler -fPIC --expt-relaxed-constexpr $extra"
nvcc $FLAGS -c -o build_$tag/mds_kernels.o mds_kernels.cu &
nvcc $FLAGS -DMDS_TU_REAL=float -DMDS_TU_KIND=1 -c -o build_$tag/rollout_float_1.o mds_rollout_tu.cu &
wait
nvcc -gencode arch=compute_100a,code=sm_100a -shared -o libmds_$tag.so build_$tag/mds_kernels.o build_$tag/rollout_float_1.o \
  build/rollout_float_0.o build/rollout_double_0.o build/rollout_double_1.o
echo built libmds_$tag.so
