#!/usr/bin/env bash
# Builds libflexgpu.so in-tree for sm_100a.  -fmad=false: fused multiply-adds are written
# explicitly (fma()) so the fp64 operation order is the one the CPU mirror oracle reproduces.
set -euo pipefail
HERE="$(cd "$(dirname "${BASH_SOURCE[0]}")" && pwd)"
OUT="${FLEXGPU_OUT:-$HERE/../flexgpu/libflexgpu.so}"
NVCC="${NVCC:-/usr/local/cuda/bin/nvcc}"
SRCS=("$HERE/flex_api.cu" "$HERE/flex_kernels.cu" "$HERE/flex_thread_kernels.cu")
[ -f "$HERE/predictor.cu" ] && SRCS+=("$HERE/predictor.cu")
[ -f "$HERE/policy.cu" ] && SRCS+=("$HERE/policy.cu")
SRCS+=("$HERE/safety.cu")
"$NVCC" --threads 0 -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -lineinfo -fmad=false \
    -Xcompiler -fPIC -shared ${NVCC_EXTRA:-} -o "$OUT" "${SRCS[@]}"
echo "built $OUT"
