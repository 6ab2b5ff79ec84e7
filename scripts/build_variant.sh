#!/bin/bash
# build_variant.sh NAME "EXTRA_NVCC_FLAGS" -> build/libporrt_NAME.so (A/B builds of the kernels; select with PORRT_B200_LIB)
set -e
cd "$(dirname "$0")/../po_rrt_b200/csrc"
mkdir -p ../../build/$1
FLAGS="-gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -fmad=false -Xcompiler -fPIC,-fvisibility=hidden,-ffp-contract=off -ccbin /usr/bin/g++"
SRCS=$(grep '^SRCS' Makefile | sed 's/SRCS := //')
for f in $SRCS; do /usr/local/cuda/bin/nvcc $FLAGS $2 -c $f -o ../../build/$1/${f%.cu}.o & done; wait
/usr/local/cuda/bin/nvcc -gencode arch=compute_100a,code=sm_100a -shared -o ../../build/libporrt_$1.so ../../build/$1/*.o -lcudart_static -lpthread -ldl -lrt
echo built build/libporrt_$1.so
