#!/usr/bin/env bash
# Builds libb200knn.so in-tree for sm_100a (cross-compiles without a GPU).
set -euo pipefail
here="$(cd "$(dirname "$0")" && pwd)"
out="$here/../lib"
mkdir -p "$out"
NVCC="${NVCC:-/usr/local/cuda/bin/nvcc}"
# EXTRA_NVCC_FLAGS / LIBNAME: experiment variants (e.g. -DB200KNN_EPI_PER_QUARTER=4)
FLAGS=(-gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xcompiler -fPIC
       --expt-relaxed-constexpr -Xptxas -v ${EXTRA_NVCC_FLAGS:-})
LIBNAME="${LIBNAME:-libb200knn.so}"
BUILD="${BUILD_DIR:-build}"
mkdir -p "$here/$BUILD"
pids=()
TC_INST="tc_inst_bf16_pair tc_inst_bf16_single tc_inst_f16_pair tc_inst_f16_single tc_inst_f16x2_pair tc_inst_f16x2_single tc_inst_bf16x3 tc_inst_tf32x3"
SRCS="$TC_INST api exact select vote prepare rescore tc_topk sharded_ops graph"
for f in $SRCS; do
  ( "$NVCC" "${FLAGS[@]}" -c "$here/$f.cu" -o "$here/$BUILD/$f.o" > "$here/$BUILD/$f.log" 2>&1 ) &
  pids+=($!)
done
rc=0
for p in "${pids[@]}"; do wait "$p" || rc=1; done
if [ $rc -ne 0 ]; then
  grep -h -E "error|Error" "$here"/$BUILD/*.log || true
  exit 1
fi
objs=()
for f in $SRCS; do objs+=("$here/$BUILD/$f.o"); done
"$NVCC" -gencode arch=compute_100a,code=sm_100a -shared -o "$out/$LIBNAME" "${objs[@]}" -cudart static
echo "built $out/$LIBNAME"
