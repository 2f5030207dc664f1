#!/bin/bash
# Builds a timing-experiment variant of the library: bnn_mlp.cu recompiled with extra -D flags, linked with the
# product's other objects into pddp_b200/lib/variants/libpddp_<name>.so (load it with PDDP_B200_LIB=<path>).
#   tools/build_variant.sh trace -DPDDP_EXP_TRACE
set -e
name=$1; shift
root=$(cd "$(dirname "$0")/.." && pwd)
src=$root/pddp_b200/csrc
out=$root/pddp_b200/lib/variants
mkdir -p $src/build/variants/$name $out
nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xcompiler -fPIC --expt-relaxed-constexpr \
     -Xptxas -v "$@" -c $src/bnn_mlp.cu -o $src/build/variants/$name/bnn_mlp.o 2> $src/build/variants/$name/ptxas.log
objs=$(ls $src/build/*.o | grep -v '/bnn_mlp.o')
nvcc -gencode arch=compute_100a,code=sm_100a -shared -o $out/libpddp_$name.so $src/build/variants/$name/bnn_mlp.o $objs
echo built $out/libpddp_$name.so
