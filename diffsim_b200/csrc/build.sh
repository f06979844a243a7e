#!/usr/bin/env bash
# Build libdiffsim_b200.so for sm_100a (cross-compiles without a GPU).
set -euo pipefail
HERE="$(cd "$(dirname "${BASH_SOURCE[0]}")" && pwd)"
OUT="${HERE}/../_lib"
OBJ="${HERE}/obj${DS_OBJ_SUFFIX:-}"
LIBNAME="${DS_LIB_NAME:-libdiffsim_b200.so}"
mkdir -p "${OUT}" "${OBJ}"
NVCC="${NVCC:-/usr/local/cuda/bin/nvcc}"
FLAGS=(-gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xcompiler -fPIC
       --expt-relaxed-constexpr -cudart static ${DS_EXTRA_NVCC_FLAGS:-})
SRCS=(ds_host.cu ds_reduce.cu ds_simmat.cu ds_qkv.cu ds_attn.cu ds_attn_bwd.cu)
pids=()
for s in "${SRCS[@]}"; do
  [ -f "${HERE}/${s}" ] || continue
  o="${OBJ}/${s%.cu}.o"
  if [ ! -f "$o" ] || [ "${HERE}/${s}" -nt "$o" ] || [ "${HERE}/ds_ptx.cuh" -nt "$o" ] || [ "${HERE}/ds_attn_common.cuh" -nt "$o" ] || [ "${HERE}/ds_gemm.cuh" -nt "$o" ] || [ "${HERE}/ds_host.h" -nt "$o" ] \
     || [ "${HERE}/../../include/diffsim_b200.h" -nt "$o" ]; then
    "${NVCC}" "${FLAGS[@]}" -Xptxas -v -c "${HERE}/${s}" -o "$o" 2> "${OBJ}/${s%.cu}.ptxas.log" &
    pids+=($!)
  fi
done
rc=0
for p in "${pids[@]:-}"; do [ -n "$p" ] && { wait "$p" || rc=1; }; done
if [ $rc -ne 0 ]; then cat "${OBJ}"/*.ptxas.log | grep -v "^ptxas info" | head -100; exit 1; fi
OBJS=()
for s in "${SRCS[@]}"; do [ -f "${OBJ}/${s%.cu}.o" ] && OBJS+=("${OBJ}/${s%.cu}.o"); done
"${NVCC}" -shared -cudart static -o "${OUT}/${LIBNAME}" "${OBJS[@]}" -Xlinker --version-script="${HERE}/exports.map"
echo "built ${OUT}/libdiffsim_b200.so"
