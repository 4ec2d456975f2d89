#!/usr/bin/env bash
# Builds vsiquantization_b200/libvsiq.so for sm_100a (nvcc cross-compiles without a GPU).
# The CUDA runtime is linked statically so the library loads with no libcudart on the path.
# Translation units compile in parallel into a scratch directory, then link.
set -euo pipefail
HERE="$(cd "$(dirname "${BASH_SOURCE[0]}")" && pwd)"
OUT="${1:-$HERE/../libvsiq.so}"
NVCC="${NVCC:-/usr/local/cuda/bin/nvcc}"
HOSTCXX="${VSIQ_HOSTCXX:-/usr/bin/g++}"
[ -x "$HOSTCXX" ] || HOSTCXX=g++
OBJ="$(mktemp -d)"
trap 'rm -rf "$OBJ"' EXIT
FLAGS=(-gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -lineinfo -ccbin "$HOSTCXX" -Xcompiler -fPIC,-O2,-Wall ${VSIQ_NVCC_EXTRA:-})
pids=()
for f in abi fake_quant observer bn_fold channels_inner multi_tensor host_pipeline peer_exchange mse_search hist_observer hist_entropy; do
    "$NVCC" "${FLAGS[@]}" -c "$HERE/$f.cu" -o "$OBJ/$f.o" &
    pids+=($!)
done
for p in "${pids[@]}"; do wait "$p"; done
"$NVCC" -gencode arch=compute_100a,code=sm_100a -ccbin "$HOSTCXX" -shared -cudart static -o "$OUT" "$OBJ"/*.o
echo "built $OUT"
