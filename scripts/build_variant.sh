#!/bin/bash
# Builds a variant of libmodfx.so with extra nvcc flags for ONE source file (kernel experiments; load it with MODFX_LIB=...).
#   scripts/build_variant.sh fc "-maxrregcount=72" variants/libmodfx_fc_r72.so
set -e
SRC=$1; FLAGS=$2; OUT=$3
ROOT=$(cd "$(dirname "$0")/.." && pwd)
python -m mod_extraction_b200._build > /dev/null
nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -Xcompiler -fPIC -I $ROOT/include -I $ROOT/mod_extraction_b200/csrc \
     $FLAGS -c $ROOT/mod_extraction_b200/csrc/$SRC.cu -o /tmp/variant_$SRC.o
OBJS=$(ls $ROOT/mod_extraction_b200/lib/obj/*.o | grep -v "/$SRC.o")
nvcc -shared -o $OUT $OBJS /tmp/variant_$SRC.o -gencode arch=compute_100a,code=sm_100a
echo built $OUT
