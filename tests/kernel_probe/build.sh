#!/bin/sh
# Builds libfocusr_probe.so (see probe.cu) for sm_100a with the product's nvcc flags (pyfocusr_b200/csrc/build.sh).
# The product's objects are reused when they are newer than every source; otherwise they are compiled here.  Output
# stays under tests/kernel_probe/.
set -e
cd "$(dirname "$0")"
NVCC=${NVCC:-/usr/local/cuda/bin/nvcc}
FLAGS="-gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -Xcompiler -fPIC -Xcompiler -fopenmp"
SRC=../../pyfocusr_b200/csrc
newest=$(ls -t $SRC/*.cu $SRC/*.cuh $SRC/*.h $SRC/*.hpp ../../include/*.h | head -n 1)
mkdir -p build
objs=""
pids=""
for f in laplacian spmm sell knn knn_pruned eigsort cpd curvature icp lsap; do
  if [ -f $SRC/build/$f.o ] && [ $SRC/build/$f.o -nt "$newest" ]; then
    objs="$objs $SRC/build/$f.o"
  else
    $NVCC $FLAGS -c $SRC/$f.cu -o build/$f.o &
    pids="$pids $!"
    objs="$objs build/$f.o"
  fi
done
$NVCC $FLAGS -c probe.cu -o build/probe.o &
pids="$pids $!"
for p in $pids; do wait $p; done
$NVCC -gencode arch=compute_100a,code=sm_100a -shared -Xlinker -Bsymbolic -o libfocusr_probe.so build/probe.o $objs -lcudart -lgomp
echo "built $(pwd)/libfocusr_probe.so"
