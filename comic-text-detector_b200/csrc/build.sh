#!/bin/bash
# Builds libctd_b200.so for sm_100a (cross-compiles without a GPU).  One object per source, compiled in
# parallel; objects live in csrc/_obj (git-ignored).
set -e
cd "$(dirname "$0")"
NVCC=${NVCC:-/usr/local/cuda/bin/nvcc}
FLAGS="-gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -Xcompiler -fPIC -Xcompiler -fvisibility=hidden"
mkdir -p _obj
pids=()
for f in engine pipeline conv_tc conv_fuse simt postproc segrep refine refine_mk resize regions group; do
  [ -f $f.cu ] || [ -f $f.cpp ] || continue
  src=$f.cu; [ -f $src ] || src=$f.cpp
  if [ ! -f _obj/$f.o ] || [ $src -nt _obj/$f.o ] || [ -n "$(find . -maxdepth 1 \( -name '*.h' -o -name '*.cuh' \) -newer _obj/$f.o)" ] \
     || [ ../../include/ctd_b200.h -nt _obj/$f.o ]; then
    $NVCC $FLAGS "$@" -c $src -o _obj/$f.o &
    pids+=($!)
  fi
done
for p in "${pids[@]}"; do wait $p; done
$NVCC -gencode arch=compute_100a,code=sm_100a -shared -o ../libctd_b200.so _obj/*.o
