#!/bin/bash
# Build libxqb200.so (sm_100a only).  -fmad=false: canonical arithmetic, see xq_common.cuh.
set -e
HERE="$(cd "$(dirname "$0")" && pwd)"
OUT="$HERE/../lib"
mkdir -p "$OUT"
# nvcc from PATH, else from the CUDA toolkit (a login shell does not put its bin/ on PATH)
command -v nvcc >/dev/null || PATH="${CUDA_HOME:-/usr/local/cuda}/bin:$PATH"
FLAGS="-gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -fmad=false --compiler-options -fPIC"
# translation units compile in parallel; an object left over from an earlier build must never be linked in place of one
# that failed to compile, so the objects go first and every compiler's exit status is checked
objs=()
for tu in vq_kernels vq_tc_kernel ms_kernels vit_kernels loss_kernels attn_kernel gemm_kernel; do objs+=("$OUT/$tu.o"); done
rm -f "${objs[@]}"
pids=()
nvcc $FLAGS -c "$HERE/vq_kernels.cu" -o "$OUT/vq_kernels.o" "$@" & pids+=($!)
nvcc $FLAGS -c "$HERE/ms_kernels.cu" -o "$OUT/ms_kernels.o" "$@" & pids+=($!)
nvcc $FLAGS -c "$HERE/vq_tc_kernel.cu" -o "$OUT/vq_tc_kernel.o" "$@" & pids+=($!)
# ViT glue kernels carry no index decisions: default contraction (-fmad=true)
nvcc ${FLAGS/-fmad=false/} -c "$HERE/vit_kernels.cu" -o "$OUT/vit_kernels.o" "$@" & pids+=($!)
nvcc ${FLAGS/-fmad=false/} -c "$HERE/loss_kernels.cu" -o "$OUT/loss_kernels.o" "$@" & pids+=($!)
nvcc ${FLAGS/-fmad=false/} -c "$HERE/attn_kernel.cu" -o "$OUT/attn_kernel.o" "$@" & pids+=($!)
nvcc ${FLAGS/-fmad=false/} -c "$HERE/gemm_kernel.cu" -o "$OUT/gemm_kernel.o" "$@" & pids+=($!)
failed=0
for p in "${pids[@]}"; do wait "$p" || failed=1; done
if [ "$failed" != 0 ]; then
    echo "build.sh: compilation failed" >&2
    exit 1
fi
nvcc -shared -o "$OUT/libxqb200.so" "${objs[@]}" -lcudart
echo "$OUT/libxqb200.so"
