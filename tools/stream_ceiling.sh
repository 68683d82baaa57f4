#!/bin/bash
# usage: tools/stream_ceiling.sh [build|run] [log2n] : builds build/stream_ceiling (sm_100a) from tools/stream_ceiling.cu,
# and with `run` (the default) runs it: one JSON line per variant on stdout
set -e
ROOT="$(cd "$(dirname "$0")/.." && pwd)"
BIN="$ROOT/build/stream_ceiling"
NVCC="${NVCC:-/usr/local/cuda/bin/nvcc}"
if [ ! -x "$BIN" ] || [ "$ROOT/tools/stream_ceiling.cu" -nt "$BIN" ] ||
   [ "$ROOT/shiftedproximaloperators.jl_b200/csrc/spx_elementwise.cuh" -nt "$BIN" ] ||
   [ "$ROOT/shiftedproximaloperators.jl_b200/csrc/spx_bulk.cuh" -nt "$BIN" ]; then
  mkdir -p "$ROOT/build"
  "$NVCC" -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -lineinfo -fmad=false -Xptxas -warn-spills \
    "$ROOT/tools/stream_ceiling.cu" -o "$BIN"
fi
[ "${1:-run}" = build ] && exit 0
exec "$BIN" "${2:-28}"
