#!/bin/bash
# Test-only: compiles the product's host-side tree builders (rz_host_bvh.hpp) on their own as host code (see hostbvh.cu).
set -e
cd "$(dirname "$0")"
mkdir -p ../_build
SO=../_build/libhostbvh.so
if [ ! -f $SO ] || [ hostbvh.cu -nt $SO ] || [ ../../rayz_b200/csrc/rz_host_bvh.hpp -nt $SO ] || [ ../../rayz_b200/csrc/rz_launch.h -nt $SO ] || [ ../../rayz_b200/csrc/rz_device.cuh -nt $SO ]; then
  nvcc -x cu -O2 -std=c++17 -shared -Xcompiler -fPIC -Wno-deprecated-gpu-targets -o $SO hostbvh.cu
fi
