#!/usr/bin/env bash
# Build liboffk.so for sm_100a in-tree (the .so travels to the GPU box with the repo snapshot).
set -euo pipefail
HERE="$(cd "$(dirname "${BASH_SOURCE[0]}")" && pwd)"
ROOT="$(cd "$HERE/../.." && pwd)"
OUT="${OFFK_OUT:-$HERE/../liboffk.so}"
ODIR="${OFFK_OBJDIR:-$HERE}"
mkdir -p "$ODIR"
NVCC="${NVCC:-/usr/local/cuda/bin/nvcc}"
FLAGS=(-O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -lineinfo -Xcompiler -fPIC -Xptxas -v
       -I"$ROOT/include" -I"$HERE" ${OFFK_EXTRA_FLAGS:-})
SRCS=(offk_api offk_gemm_tc offk_gemm_tma offk_stencil offk_head offk_train)
OBJS=()
PIDS=()
for f in "${SRCS[@]}"; do
  [ -f "$HERE/$f.cu" ] || continue
  "$NVCC" "${FLAGS[@]}" -c "$HERE/$f.cu" -o "$ODIR/$f.o" 2> "$ODIR/$f.ptxas.log" &      # one nvcc per translation unit, in parallel
  PIDS+=("$!:$f")
  OBJS+=("$ODIR/$f.o")
done
FAILED=0
for pf in "${PIDS[@]}"; do
  if ! wait "${pf%%:*}"; then
    cat "$ODIR/${pf##*:}.ptxas.log" >&2
    FAILED=1
  fi
done
[ "$FAILED" = 0 ] || exit 1
"$NVCC" -shared -o "$OUT" "${OBJS[@]}" -gencode arch=compute_100a,code=sm_100a -lcudart
echo "built $OUT"
