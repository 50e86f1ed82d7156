#!/bin/bash
# Compile the CUDA library to a scratch .so with ptxas statistics for kernels matching $1.  The flags are the
# library's own (_lib.NVCC_FLAGS): with -split-compile the code of a kernel depends on the rest of the translation
# unit, so statistics from other flags describe a different binary.
cd "$(dirname "$0")/.." || exit 1
FLAGS=$(python3 -c 'import importlib.util as u; s = u.spec_from_file_location("l", "ris_vec_marl_b200/_lib.py"); m = u.module_from_spec(s); s.loader.exec_module(m); print(" ".join(m.NVCC_FLAGS))') || exit 1
OUT=$(mktemp -d) || exit 1
trap 'rm -rf "$OUT"' EXIT
cd ris_vec_marl_b200/csrc || exit 1
nvcc $FLAGS -o "$OUT/librisvec.so" risvec.cu -Xptxas -v 2>&1 | grep -E "error|$1" -A2 | grep -E "error|Compiling|registers|spill"
