#!/bin/bash
# Builds libb200nuts.so for sm_100a in-tree (travels to the GPU box with the snapshot).
set -e
cd "$(dirname "$0")"
NVCC=${NVCC:-/usr/local/cuda/bin/nvcc}
$NVCC -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xcompiler -fPIC -shared \
  ${B200_PTXAS_V:+-Xptxas -v} \
  -o ${B200_OUT:-pymc_b200/libb200nuts.so} pymc_b200/csrc/b200nuts.cu
echo "built pymc_b200/libb200nuts.so"
