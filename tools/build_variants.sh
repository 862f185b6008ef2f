#!/bin/bash
# Builds tuning variants of the batched kernels into tools/variants/ (N=4,6 only).
# usage: tools/build_variants.sh name "-DFLAG=.. -DFLAG=.." [name flags]...
set -e
cd "$(dirname "$0")/.."
mkdir -p tools/variants
C=bounded_lsq_b200/csrc
NV="nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -lineinfo -fmad=false
    -Xcompiler -fPIC -Xptxas -v -DBLSQ_ONLY_N46"
while [ $# -gt 1 ]; do
  name=$1; flags=$2; shift 2
  V=tools/variants/$name
  ($NV $flags -DBLSQ_N=4 -c $C/blsq_batched_n.cu -o ${V}_n4.o 2> $V.ptxas.log &&
   $NV $flags -DBLSQ_N=6 -c $C/blsq_batched_n.cu -o ${V}_n6.o 2>> $V.ptxas.log &&
   $NV $flags -shared $C/blsq_batched.cu $C/blsq_elementwise.cu ${V}_n4.o ${V}_n6.o \
     -o tools/variants/lib_$name.so -lcudart 2>> $V.ptxas.log && echo built $name) &
done
wait
