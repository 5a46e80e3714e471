#!/usr/bin/env bash
# Builds libunmore_b200.so (sm_100a only) next to the package so it travels with the repo snapshot.
set -euo pipefail
HERE="$(cd "$(dirname "${BASH_SOURCE[0]}")" && pwd)"
OUT="${UNMORE_OUT:-${HERE}/../libunmore_b200.so}"   # UNMORE_OUT: a second build beside the first, for A/B runs
NVCC="${NVCC:-/usr/local/cuda/bin/nvcc}"
FLAGS=(-gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xcompiler -fPIC,-O3,-Wall
       --expt-relaxed-constexpr -Xptxas -v -shared -cudart static)
"${NVCC}" "${FLAGS[@]}" -o "${OUT}" "${HERE}"/*.cu 2> "${OUT%.so}_build.log" || { cat "${OUT%.so}_build.log" >&2; exit 1; }
echo "built ${OUT}"
