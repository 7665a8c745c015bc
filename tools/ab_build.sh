#!/bin/bash
# Development aid: build the working tree's warp_fast.cu, linked with the other objects of the last
# make, as the named library variant tools/_ab/<name>.so for same-box A/B runs (tools/ab_run.sh,
# tools/kbench.py --lib).   tools/ab_build.sh name [nvcc flags]
set -e
cd "$(dirname "$0")/../bev_b200/csrc"
name=$1; shift
NV="/usr/local/cuda/bin/nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -lineinfo -fmad=false -Xcompiler -fPIC,-ffp-contract=off,-Wall -Xptxas -v --expt-relaxed-constexpr"
mkdir -p ../../tools/_ab
$NV "$@" -c warp_fast.cu -o ../../tools/_ab/$name.o 2> ../../tools/_ab/$name.ptxas.log || { cat ../../tools/_ab/$name.ptxas.log; exit 1; }
# every other object of the Makefile's SRCS, as the last make left it
objs=$(sed -n 's/^SRCS *= *//p' Makefile | tr ' ' '\n' | grep -v '^warp_fast.cu$' | sed 's/\.cu$/.o/')
/usr/local/cuda/bin/nvcc -gencode arch=compute_100a,code=sm_100a -shared -o ../../tools/_ab/$name.so ../../tools/_ab/$name.o $objs
grep -A1 "PxU8C3Lb1ELi6ELi4" ../../tools/_ab/$name.ptxas.log | grep -E "registers|spill" | head -3
