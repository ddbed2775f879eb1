#!/bin/bash
# Build an A/B variant of libljmd.so with extra nvcc flags into variants/NAME/ (git-ignored, travels
# with gpurun); select it at run time with LJMD_LIB=variants/NAME/libljmd.so.
#   scripts/build_variant.sh debug -DLJMD_DEBUG_CHECKS
set -e
ROOT=$(cd "$(dirname "$0")/.." && pwd)
NAME=$1; shift
OUT=$ROOT/variants/$NAME
mkdir -p "$OUT"
CSRC=$ROOT/jax_tpus_benchmark_physics_simulation_b200/csrc
for f in api allpairs cells dist pairlaw probe; do
  nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -lineinfo -Xcompiler -fPIC,-O2 "$@" \
       -c "$CSRC/$f.cu" -o "$OUT/$f.o" &
done
wait
nvcc -gencode arch=compute_100a,code=sm_100a -shared -o "$OUT/libljmd.so" "$OUT"/*.o -lcudart -ldl
rm -f "$OUT"/*.o
echo "$OUT/libljmd.so"
