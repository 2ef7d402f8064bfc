#!/bin/bash
# Builds dang_b200/libdang_gpu.so for sm_100a (cross-compiles without a GPU).
# One object per translation unit, compiled in parallel, then one link.
set -euo pipefail
here="$(cd "$(dirname "$0")" && pwd)"
out="$here/../libdang_gpu.so"
obj="$here/_obj"
mkdir -p "$obj"
NVCC="${NVCC:-/usr/local/cuda/bin/nvcc}"
FLAGS=(-std=c++17 -O3 -lineinfo -gencode arch=compute_100a,code=sm_100a -Xcompiler -fPIC,-O2,-Wall "$@")
units=(dang_gpu host_cg host_tmpl host_data host_mh_pp host_mh_ppd2 host_mh_ppd3 host_mh_ppd5 host_mh_ppd8 host_mh_ppf host_mh_ppx host_mh_fs host_udgrade host_post)
declare -A deps=(
  [dang_gpu]="kernels_data.cuh"
  [host_cg]="kernels_cg.cuh kernels_cg_solve.cuh kernels_uni.cuh kernels_stream.cuh"
  [host_tmpl]="kernels_tmpl.cuh"
  [host_data]="kernels_data.cuh kernels_uni.cuh"
  [host_mh_pp]="kernels_mh.cuh"
  [host_mh_ppf]="kernels_mh.cuh kernels_mh_fast.cuh"
  [host_udgrade]=""
  [host_post]="kernels_post.cuh kernels_data.cuh"
  [host_mh_ppd2]="kernels_mh.cuh host_mh_ppd.inc"
  [host_mh_ppd3]="kernels_mh.cuh host_mh_ppd.inc"
  [host_mh_ppd5]="kernels_mh.cuh host_mh_ppd.inc"
  [host_mh_ppd8]="kernels_mh.cuh host_mh_ppd.inc"
  [host_mh_ppx]="kernels_mh.cuh kernels_mh_fast.cuh kernels_mh_pix.cuh"
  [host_mh_fs]="kernels_mh.cuh kernels_uni.cuh kernels_stream.cuh kernels_cg.cuh"
)
pids=()
for u in "${units[@]}"; do
  # rebuild a unit when its source, one of its headers or this script is newer than its object
  stale=0
  [ -f "$obj/$u.o" ] || stale=1
  for d in "$u.cu" host.cuh common.cuh build.sh ../../include/dang_gpu.h ${deps[$u]}; do
    [ "$here/$d" -nt "$obj/$u.o" ] && stale=1
  done
  if [ "$stale" = 1 ]; then
    "$NVCC" "${FLAGS[@]}" -c "$here/$u.cu" -o "$obj/$u.o" &
    pids+=($!)
  fi
done
for p in "${pids[@]:-}"; do [ -n "$p" ] && wait "$p"; done
objs=()
for u in "${units[@]}"; do objs+=("$obj/$u.o"); done
"$NVCC" -shared -gencode arch=compute_100a,code=sm_100a -o "$out" "${objs[@]}" -ldl
echo "built $out"
