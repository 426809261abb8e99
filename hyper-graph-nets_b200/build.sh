#!/usr/bin/env bash
# Build libhgn_b200.so (sm_100a only) in-tree: hyper-graph-nets_b200/hgn_b200/libhgn_b200.so
set -euo pipefail
cd "$(dirname "$0")"
NVCC=${NVCC:-/usr/local/cuda/bin/nvcc}
OUT=hgn_b200/libhgn_b200.so
mkdir -p build
FLAGS=(-gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xcompiler -fPIC -Xptxas -v --threads 0)
objs=()
pids=()
for f in csrc/cabi.cu csrc/segment.cu csrc/mlp_f32.cu csrc/mlp_tc.cu csrc/edge_tc.cu csrc/edge_fwd_tc.cu csrc/world_edges.cu csrc/peer.cu csrc/io_mlp_tc.cu csrc/segment_long.cu; do
  o=build/$(basename "${f%.cu}").o
  objs+=("$o")
  if [[ ! -f "$o" || "$f" -nt "$o" || csrc/common.cuh -nt "$o" || csrc/tc05.cuh -nt "$o" || csrc/tile_common.cuh -nt "$o" || ../include/hgn_b200.h -nt "$o" ]]; then
    "$NVCC" "${FLAGS[@]}" -c "$f" -o "$o" > "build/$(basename "${f%.cu}").log" 2>&1 &
    pids+=($!)
  fi
done
for p in "${pids[@]:-}"; do [[ -n "$p" ]] && wait "$p"; done
"$NVCC" -shared -o "$OUT" "${objs[@]}" -lcudart
echo "built $OUT"
