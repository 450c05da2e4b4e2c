#!/bin/bash
# Build libxqb200.so (sm_100a only).  -fmad=false: canonical arithmetic, see xq_common.cuh.
set -e
HERE="$(cd "$(dirname "$0")" && pwd)"
OUT="$HERE/../lib"
mkdir -p "$OUT"
# nvcc from PATH, else from the CUDA toolkit (a login shell does not put its bin/ on PATH)
command -v nvcc >/dev/null || PATH="${CUDA_HOME:-/usr/local/cuda}/bin:$PATH"
FLAGS="-gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -fmad=false --compiler-options -fPIC"
nvcc $FLAGS -c "$HERE/vq_kernels.cu" -o "$OUT/vq_kernels.o" "$@" &
nvcc $FLAGS -c "$HERE/ms_kernels.cu" -o "$OUT/ms_kernels.o" "$@" &
nvcc $FLAGS -c "$HERE/vq_tc_kernel.cu" -o "$OUT/vq_tc_kernel.o" "$@" &
# ViT glue kernels carry no index decisions: default contraction (-fmad=true)
nvcc ${FLAGS/-fmad=false/} -c "$HERE/vit_kernels.cu" -o "$OUT/vit_kernels.o" "$@" &
nvcc ${FLAGS/-fmad=false/} -c "$HERE/loss_kernels.cu" -o "$OUT/loss_kernels.o" "$@" &
nvcc ${FLAGS/-fmad=false/} -c "$HERE/attn_kernel.cu" -o "$OUT/attn_kernel.o" "$@" &
nvcc ${FLAGS/-fmad=false/} -c "$HERE/gemm_kernel.cu" -o "$OUT/gemm_kernel.o" "$@" &
wait
nvcc -shared -o "$OUT/libxqb200.so" "$OUT/vq_kernels.o" "$OUT/vq_tc_kernel.o" "$OUT/ms_kernels.o" "$OUT/vit_kernels.o" "$OUT/loss_kernels.o" "$OUT/attn_kernel.o" "$OUT/gemm_kernel.o" -lcudart
echo "$OUT/libxqb200.so"
