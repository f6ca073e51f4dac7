#!/bin/bash
# Build a tuning variant of libgingr_cuda.so:  tools/build_variant.sh NAME file.cu "-DFOO=1 -DBAR=2"
# -> gingr_b200/lib/variants/libgingr_cuda_NAME.so (all other objects are reused from the main build)
set -e
NAME=$1; SRC=$2; FLAGS=$3
cd "$(dirname "$0")/.."
mkdir -p gingr_b200/lib/variants
EXTRA=""
[ "$SRC" = "closest.cu" ] && EXTRA="-fmad=false"
[ "$SRC" = "grid.cu" ] && EXTRA="-fmad=false"
nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -lineinfo -Xcompiler -fPIC,-fvisibility=hidden -Xptxas -v $EXTRA $FLAGS \
  -c gingr_b200/csrc/$SRC -o gingr_b200/lib/variants/${SRC%.cu}_$NAME.o 2> gingr_b200/lib/variants/${SRC%.cu}_$NAME.log
OBJS=$(ls gingr_b200/lib/obj/*.o | grep -v "/${SRC%.cu}.o")
nvcc -gencode arch=compute_100a,code=sm_100a -shared -o gingr_b200/lib/variants/libgingr_cuda_$NAME.so $OBJS gingr_b200/lib/variants/${SRC%.cu}_$NAME.o -ldl
grep -A2 "estep_colsum\|estep_rowsum" gingr_b200/lib/variants/${SRC%.cu}_$NAME.log | grep "Used" | tr '\n' ' '; echo
