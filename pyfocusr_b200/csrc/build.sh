#!/bin/sh
# Builds libfocusr_b200.so in-tree for sm_100a (B200).  nvcc cross-compiles without a GPU.
set -e
cd "$(dirname "$0")"
NVCC=${NVCC:-/usr/local/cuda/bin/nvcc}
FLAGS="-gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -Xcompiler -fPIC -Xcompiler -fopenmp"
mkdir -p build
pids=""
for f in laplacian spmm sell eigs knn knn_pruned eigsort cpd curvature icp lsap features shape surface; do
  EXTRA=""
  # surface.cu: its pruned search and its brute-force reference must score a (query, triangle) pair bit for bit alike,
  # and where the compiler fuses a multiply and an add into an FMA depends on the kernel the code is inlined into
  [ $f = surface ] && EXTRA="-fmad=false"
  $NVCC $FLAGS $EXTRA -c $f.cu -o build/$f.o &
  pids="$pids $!"
done
for p in $pids; do wait $p; done
$NVCC -gencode arch=compute_100a,code=sm_100a -shared -o libfocusr_b200.so build/laplacian.o build/spmm.o build/sell.o build/eigs.o build/knn.o build/knn_pruned.o build/eigsort.o build/cpd.o build/curvature.o build/icp.o build/lsap.o build/features.o build/shape.o build/surface.o -lcudart -lgomp
echo "built $(pwd)/libfocusr_b200.so"
