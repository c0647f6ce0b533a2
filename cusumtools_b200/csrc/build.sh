#!/bin/bash
# Builds libcusumtools_b200.so for sm_100a in-tree (the .so travels to the GPU box).
set -e
cd "$(dirname "$0")"
NVCC=${NVCC:-/usr/local/cuda/bin/nvcc}
FLAGS="-gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -Xcompiler -fPIC -I../../include ${CT_EXTRA_NVCC_FLAGS}"
OBJS=""
PIDS=""
for f in ct_api ct_filter ct_filter_seq ct_detect ct_cusum ct_stepfit ct_welch ct_loader; do
  if [ ! -f $f.o ] || [ $f.cu -nt $f.o ] || [ ct_common.cuh -nt $f.o ] || [ ../../include/cusumtools_b200.h -nt $f.o ]; then
    # a failed compile must not leave a stale object behind for the link step
    ( rm -f $f.o; $NVCC $FLAGS -c $f.cu -o $f.o.tmp && mv $f.o.tmp $f.o ) &
    PIDS="$PIDS $!"
  fi
  OBJS="$OBJS $f.o"
done
FAIL=0
for p in $PIDS; do wait $p || FAIL=1; done
rm -f ./*.o.tmp
if [ $FAIL -ne 0 ]; then echo "build.sh: compilation failed" >&2; exit 1; fi
$NVCC -shared -gencode arch=compute_100a,code=sm_100a -o ../libcusumtools_b200.so $OBJS -lcudart
echo "built $(cd .. && pwd)/libcusumtools_b200.so"
