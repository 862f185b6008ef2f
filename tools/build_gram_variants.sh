#!/bin/bash
# Builds tuning variants of the n = 64 Gram kernels into tools/variants/.
# usage: tools/build_gram_variants.sh name "-DBLSQ_G8_CW=.. ..." [name flags]...
# every variant must define ALL of BLSQ_G8_{CW,ROLES,CG,S1,S2,YB2}
set -e
cd "$(dirname "$0")/.."
mkdir -p tools/variants
C=bounded_lsq_b200/csrc
NV="nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -lineinfo -fmad=false
    -Xcompiler -fPIC -Xptxas -v -DBLSQ_ONLY_N46"
while [ $# -gt 1 ]; do
  name=$1; flags=$2; shift 2
  V=tools/variants/g_$name
  ($NV $flags -DBLSQ_N=4 -c $C/blsq_batched_n.cu -o ${V}_n4.o 2> $V.ptxas.log &&
   $NV $flags -DBLSQ_N=6 -c $C/blsq_batched_n.cu -o ${V}_n6.o 2>> $V.ptxas.log &&
   $NV $flags -shared $C/blsq_batched.cu $C/blsq_elementwise.cu $C/blsq_models.cu \
     $C/blsq_tall_gram.cu $C/blsq_tall_factor.cu $C/blsq_tall_round.cu ${V}_n4.o ${V}_n6.o \
     -o tools/variants/libg_$name.so -lcudart 2>> $V.ptxas.log && echo built $name) &
done
wait
