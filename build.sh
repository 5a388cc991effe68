#!/bin/bash
# Builds libyuki_gpu.so (host helpers + sm_100a kernels) in-tree and the oracle's liboracle.so.
set -e
cd "$(dirname "$0")"
NVCC=${NVCC:-/usr/local/cuda/bin/nvcc}
SRC=yuki_b200/csrc
OUT=yuki_b200/libyuki_gpu.so
$NVCC -std=c++17 -O3 -gencode arch=compute_100a,code=sm_100a -lineinfo \
  --fmad=false -prec-div=true -prec-sqrt=true -ftz=false \
  -Xcompiler -fPIC,-ffp-contract=off,-fno-fast-math,-pthread,-Wall \
  -Iinclude -I$SRC -shared -o $OUT \
  $SRC/render.cu $SRC/host_scene.cpp $SRC/host_bvh.cpp $SRC/host_ply.cpp $SRC/host_exr.cpp $SRC/host_pbrt.cpp $SRC/host_mitsuba.cpp $SRC/post.cu $SRC/denoise.cu -lz ${YK_NVCC_EXTRA}
make -s -C oracle
echo "built $OUT and oracle/liboracle.so"
