#!/usr/bin/env bash
# Build libparrm_b200.so in-tree for sm_100a (nvcc cross-compiles without a GPU).
set -euo pipefail
here="$(cd "$(dirname "${BASH_SOURCE[0]}")" && pwd)"
root="$(cd "$here/../.." && pwd)"
out="$here/../libparrm_b200.so"
obj="$here/build"
mkdir -p "$obj"
NVCC="${NVCC:-/usr/local/cuda/bin/nvcc}"
FLAGS=(-gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17
       -Xcompiler -fPIC -I"$root/include" -I"$here" -I"$obj" ${PARRM_NVCC_EXTRA:-})
# The run-time specialised filter kernel travels inside the library as source text
# (filter_jit.cu hands it to NVRTC); the same file is also compiled here with its default
# parameters so that a syntax or resource error shows up at build time.
{ printf 'R"PARRMSRC('; cat "$here/filter_comb_e.cuh"; printf ')PARRMSRC"\n'; } > "$obj/filter_comb_e_src.inc"
SRCS=(cabi taps filter filter_plan filter_jit standardise period_eval psd neldermead host_copy stream transpose)
pids=()
for src in "${SRCS[@]}"; do
  "$NVCC" "${FLAGS[@]}" -c "$here/$src.cu" -o "$obj/$src.o" &
  pids+=($!)
done
"$NVCC" "${FLAGS[@]}" -Xptxas -v -c "$here/filter_comb_e_check.cu" -o "$obj/filter_comb_e_check.o" \
        2> "$obj/filter_comb_e_check.ptxas.txt" &
pids+=($!)
for pid in "${pids[@]}"; do wait "$pid"; done
objs=()
for src in "${SRCS[@]}"; do objs+=("$obj/$src.o"); done
"$NVCC" -gencode arch=compute_100a,code=sm_100a -shared -o "$out" "${objs[@]}" -cudart static -ldl
echo "built $out"
