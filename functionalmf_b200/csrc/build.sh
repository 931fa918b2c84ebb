#!/bin/bash
# Build libbtf_b200.so for sm_100a in-tree (travels to the GPU box with gpurun).
set -e
HERE="$(cd "$(dirname "$0")" && pwd)"
OUT="$HERE/../libbtf_b200.so"
NVCC=${NVCC:-/usr/local/cuda/bin/nvcc}
FLAGS="-std=c++17 -O3 -lineinfo -gencode arch=compute_100a,code=sm_100a -Xcompiler -fPIC -Xptxas -v"
mkdir -p "$HERE/_obj"
SRCS="engine stats_kernels stats_zpre solve_kernels band_lookahead hyper_kernels pg_kernels gass_kernels eval_kernels i8gemm2 stats_i8 nccl_shard peaks"
pids=()
for f in $SRCS; do
  ( $NVCC $FLAGS -c "$HERE/$f.cu" -o "$HERE/_obj/$f.o" > "$HERE/_obj/$f.log" 2>&1 || { cat "$HERE/_obj/$f.log"; exit 1; } ) &
  pids+=($!)
done
rc=0
for p in "${pids[@]}"; do wait $p || rc=1; done
[ $rc -eq 0 ] || exit 1
# the objects of this source list only: _obj/ may still hold those of a source that has since been removed or renamed
( cd "$HERE/_obj" && $NVCC -shared -o "$OUT" $(printf '%s.o ' $SRCS) -ldl )
echo "built $OUT"
