#!/bin/bash
# Bounds-checked build of the library (-DCT_BOUNDS_CHECK: every hand-computed workspace offset is checked on the device,
# a violation prints the site and traps) into build_ab/libcusumtools_b200_checked.so; run the GPU tests against it with
#   CT_LIB_PATH=build_ab/libcusumtools_b200_checked.so python -m pytest tests -m gpu -q
set -e
cd "$(dirname "$0")/../cusumtools_b200/csrc"
NVCC=${NVCC:-/usr/local/cuda/bin/nvcc}
OUT=../../build_ab
mkdir -p $OUT/checked
FLAGS="-gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -Xcompiler -fPIC -I../../include -DCT_BOUNDS_CHECK"
PIDS=""
for f in ct_api ct_filter ct_filter_seq ct_detect ct_cusum ct_stepfit ct_welch ct_loader; do
  ( $NVCC $FLAGS -c $f.cu -o $OUT/checked/$f.o ) &
  PIDS="$PIDS $!"
done
FAIL=0
for p in $PIDS; do wait $p || FAIL=1; done
if [ $FAIL -ne 0 ]; then echo "build_checked.sh: compilation failed" >&2; exit 1; fi
$NVCC -shared -gencode arch=compute_100a,code=sm_100a -o $OUT/libcusumtools_b200_checked.so $OUT/checked/*.o -lcudart
echo "built $OUT/libcusumtools_b200_checked.so"
