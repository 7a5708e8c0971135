#!/usr/bin/env bash
# Builds the CUDA extension in-tree for sm_100a (nvcc cross-compiles without a GPU).
#   build.sh            -> libcdc_b200.so        the product (fp16 storage, no environment switches, no tools hooks)
#   build.sh bf16       -> libcdc_b200_bf16.so   same sources with -DCDC_ACT_FP16=0: the bf16 variant the precision tests measure
#   build.sh tools      -> libcdc_b200_tools.so  -DCDC_TOOLS: graph-skip hook (CDC_GRAPH_SKIP), flushed conv timing (CDC_TEST_CONV_REPS), barrier-timeout messages
#   build.sh all        -> all three
set -euo pipefail
HERE="$(cd "$(dirname "${BASH_SOURCE[0]}")" && pwd)"
NVCC="${NVCC:-/usr/local/cuda/bin/nvcc}"
SRCS=(conv_tc conv_kf elementwise attention entropy rans runner bitstream)

build_variant() {  # name, extra flags...
  local name="$1"; shift
  local suffix=""; [ "${name}" != "product" ] && suffix="_${name}"
  local OUT="${HERE}/../libcdc_b200${suffix}.so"
  local OBJ="${HERE}/../build${suffix}"
  local FLAGS=(-gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xcompiler -fPIC -Xcompiler -fvisibility=default "$@")
  mkdir -p "${OBJ}"
  local pids=() objs=()
  for f in "${SRCS[@]}"; do
    objs+=("${OBJ}/${f}.o")
    if [ ! -f "${OBJ}/${f}.o" ] || [ "${HERE}/${f}.cu" -nt "${OBJ}/${f}.o" ] || [ "${HERE}/build.sh" -nt "${OBJ}/${f}.o" ] || [ -n "$(find "${HERE}" "${HERE}/../../include" \( -name '*.cuh' -o -name '*.h' \) -newer "${OBJ}/${f}.o" 2>/dev/null | head -1)" ]; then
      "${NVCC}" "${FLAGS[@]}" -c "${HERE}/${f}.cu" -o "${OBJ}/${f}.o" &
      pids+=($!)
    fi
  done
  local rc=0
  for p in "${pids[@]:-}"; do [ -n "$p" ] && { wait "$p" || rc=1; }; done
  [ "${rc}" = 0 ] || { echo "compile failed (${name})" >&2; return 1; }
  "${NVCC}" -gencode arch=compute_100a,code=sm_100a -shared -o "${OUT}" "${objs[@]}"
  echo "built ${OUT}"
}

what="${1:-product}"
case "${what}" in
  product) build_variant product ;;
  bf16)    build_variant bf16 -DCDC_ACT_FP16=0 ;;
  tools)   build_variant tools -DCDC_TOOLS ;;
  all)     build_variant product & p1=$!; build_variant bf16 -DCDC_ACT_FP16=0 & p2=$!; build_variant tools -DCDC_TOOLS & p3=$!
           wait $p1; wait $p2; wait $p3 ;;
  *) echo "usage: build.sh [product|bf16|tools|all]" >&2; exit 2 ;;
esac
