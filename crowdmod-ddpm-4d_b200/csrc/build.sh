#!/usr/bin/env bash
# Builds libcrowdmod_b200.so (sm_100a only) next to the Python package.  Called by
# __graft_entry__.build(); safe to run by hand.  cudart is linked statically and the driver
# API is resolved at run time (cudaGetDriverEntryPoint), so the library loads on a CPU-only
# box for the symbol-export tests.
set -euo pipefail
HERE="$(cd "$(dirname "${BASH_SOURCE[0]}")" && pwd)"
OUT="${HERE}/../libcrowdmod_b200.so"
NVCC="${NVCC:-/usr/local/cuda/bin/nvcc}"
FLAGS=(-gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -lineinfo
       -Xcompiler -fPIC -Xcompiler -fvisibility=hidden --expt-relaxed-constexpr
       -cudart static)
OBJ="${HERE}/build"
mkdir -p "${OBJ}"
pids=()
for f in api conv_umma kernels unet backward feed_metrics dit attn_long; do
  if [[ ! -f "${OBJ}/${f}.o" || "${HERE}/${f}.cu" -nt "${OBJ}/${f}.o" || -n "$(find "${HERE}" -name '*.cuh' -newer "${OBJ}/${f}.o" 2>/dev/null)" || "${HERE}/../../include/crowdmod_b200.h" -nt "${OBJ}/${f}.o" ]]; then
    "${NVCC}" "${FLAGS[@]}" ${CM_PTXAS_V:+-Xptxas -v} -c "${HERE}/${f}.cu" -o "${OBJ}/${f}.o" &
    pids+=($!)
  fi
done
for p in "${pids[@]:-}"; do [[ -n "$p" ]] && wait "$p"; done
"${NVCC}" "${FLAGS[@]}" -shared -o "${OUT}" "${OBJ}"/api.o "${OBJ}"/conv_umma.o "${OBJ}"/kernels.o "${OBJ}"/unet.o "${OBJ}"/backward.o "${OBJ}"/feed_metrics.o "${OBJ}"/dit.o "${OBJ}"/attn_long.o
echo "built ${OUT}"
