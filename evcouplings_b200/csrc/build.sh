#!/bin/bash
# Build libevcplm.so in-tree for sm_100a (no GPU needed: nvcc cross-compiles).
set -e
cd "$(dirname "$0")"
NVCC=${NVCC:-/usr/local/cuda/bin/nvcc}
FLAGS="-gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xcompiler -fPIC -Xptxas -v"
mkdir -p _obj
for f in api hamming plm_gather plm_tc model_ops vecops fit a2m_reader mean_field; do
  if [ ! -f _obj/$f.o ] || [ $f.cu -nt _obj/$f.o ] || [ common.cuh -nt _obj/$f.o ] || [ internal.h -nt _obj/$f.o ] || [ ../../include/evcplm.h -nt _obj/$f.o ]; then
    $NVCC $FLAGS -c $f.cu -o _obj/$f.o 2> _obj/$f.ptxas.log || { cat _obj/$f.ptxas.log; exit 1; }
  fi
done
$NVCC -gencode arch=compute_100a,code=sm_100a -shared -o libevcplm.so _obj/api.o _obj/hamming.o _obj/plm_gather.o _obj/plm_tc.o _obj/model_ops.o _obj/vecops.o _obj/fit.o _obj/a2m_reader.o _obj/mean_field.o
echo "built $(pwd)/libevcplm.so"
