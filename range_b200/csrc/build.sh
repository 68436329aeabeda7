#!/bin/bash
# Builds range_b200/librange_b200.so for sm_100a (no GPU needed: nvcc cross-compiles).
set -euo pipefail
cd "$(dirname "$0")"
NVCC=${NVCC:-/usr/local/cuda/bin/nvcc}
# --use_fast_math only affects fp32 intrinsics; every fp64 path (SH, SIREN) is unaffected.
FLAGS="-gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -Xcompiler -fPIC --use_fast_math -diag-suppress 177"
mkdir -p ../../build
pids=()
for f in encoder encoder_tc encoder_raster retrieval retrieval_pc topk sort merge capi; do
  $NVCC $FLAGS ${NVCC_EXTRA:-} -c $f.cu -o ../../build/$f.o &
  pids+=($!)
done
${CXX:-g++} -O3 -std=c++17 -fPIC -pthread -c host.cpp -o ../../build/host.o &
pids+=($!)
for p in "${pids[@]}"; do wait $p; done
$NVCC -arch=sm_100a -shared -cudart static -o ../librange_b200.so ../../build/encoder.o ../../build/encoder_tc.o ../../build/encoder_raster.o ../../build/retrieval.o ../../build/retrieval_pc.o ../../build/topk.o ../../build/sort.o ../../build/merge.o ../../build/capi.o ../../build/host.o -Xlinker -lpthread
echo "built $(cd .. && pwd)/librange_b200.so"
