#!/bin/bash
# Builds libfastnn.so in-tree for sm_100a.  --fmad=false: the reference is Java (no FMA
# contraction) and the circular ordering must be bit-exact.
set -e
cd "$(dirname "$0")"
SRC=fastneighbornet_b200/csrc
OUT=${FNN_OUT:-fastneighbornet_b200/libfastnn.so}
nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -lineinfo --fmad=false -prec-div=true -prec-sqrt=true \
     -Xcompiler -fPIC -Xcompiler -Wno-deprecated-declarations -shared -Iinclude -I$SRC ${NVCC_EXTRA} \
     -o $OUT $SRC/fnn_order.cu $SRC/fnn_host.cu $SRC/fnn_csw.cu $SRC/fnn_phylip.cpp $SRC/fnn_nexus.cpp \
     $SRC/fnn_dist.cu $SRC/fnn_align.cpp $SRC/fnn_boot.cu
echo "built $OUT"
