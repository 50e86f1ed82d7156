#!/bin/bash
# Compile the CUDA library to a scratch .so with ptxas statistics for kernels matching $1
cd "$(dirname "$0")/../ris_vec_marl_b200/csrc" || exit 1
nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xcompiler -fPIC -shared \
     -o /tmp/librisvec.so risvec.cu -Xptxas -v 2>&1 | grep -E "error|$1" -A2 | grep -E "error|Compiling|registers|spill"
