#!/bin/bash
# Build libvfeat.so in-tree for sm_100a (nvcc cross-compiles without a GPU).
set -e
cd "$(dirname "$0")"
SRC=video_features_b200/csrc
nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -shared -Xcompiler -fPIC \
     -o video_features_b200/libvfeat.so $SRC/gemm.cu $SRC/attn_gemm.cu $SRC/kernels.cu $SRC/host.cu $SRC/clip.cu $SRC/i3d.cu $SRC/i3d_kernels.cu $SRC/raft.cu $SRC/raft_kernels.cu \
     $SRC/conv2d.cu $SRC/resnet.cu $SRC/resnet_kernels.cu "$@"
