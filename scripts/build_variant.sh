#!/bin/bash
# build a library variant for A/B runs on the GPU box: scripts/build_variant.sh NAME [-DFLAG=V ...]
# -> build/variants/libfwgym_NAME.so (select with FWGYM_LIB=..., scripts/gpu_ab.sh)
NAME=$1; shift
mkdir -p build/variants
nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 --shared -Xcompiler -fPIC "$@" \
  -o build/variants/libfwgym_$NAME.so fixed-wing-gym_b200/csrc/fwgym.cu && echo built build/variants/libfwgym_$NAME.so
