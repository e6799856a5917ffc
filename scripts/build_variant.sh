#!/bin/bash
# usage: scripts/build_variant.sh NAME -DFLAG[=V] ...   -> translation_transformer_b200/libttb200_NAME.so
# Experimental build of the same sources with extra nvcc flags, selected at run time with TTB_LIB=libttb200_NAME.so (A/B runs).
set -e
NAME=$1; shift
cd "$(dirname "$0")/../translation_transformer_b200"
# the sources of the library, as build.py compiles them
SOURCES=$(python3 -c "from build import SOURCES; print(' '.join(SOURCES))")
mkdir -p csrc/build_$NAME
pids=()
for f in $SOURCES; do
  nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xcompiler -fPIC --expt-relaxed-constexpr "$@" -c csrc/$f -o csrc/build_$NAME/$f.o &
  pids+=($!)
done
for p in "${pids[@]}"; do wait $p; done
nvcc -gencode arch=compute_100a,code=sm_100a -shared -o libttb200_$NAME.so csrc/build_$NAME/*.o -lcudart
echo built libttb200_$NAME.so
