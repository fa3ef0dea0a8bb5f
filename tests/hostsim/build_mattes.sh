#!/bin/bash
# Test-only: compiles the ID mattes' rank key (rz_device.cuh's rz_matte_key) as host code (see mattes.cu).
set -e
cd "$(dirname "$0")"
mkdir -p ../_build
SO=../_build/libhostmatte.so
if [ ! -f $SO ] || [ mattes.cu -nt $SO ] || [ ../../rayz_b200/csrc/rz_sampler.cuh -nt $SO ] || [ ../../rayz_b200/csrc/rz_device.cuh -nt $SO ] || [ ../../include/rayz_cuda.h -nt $SO ]; then
  nvcc -x cu -O2 -std=c++17 -shared -Xcompiler -fPIC -Wno-deprecated-gpu-targets -o $SO mattes.cu
fi
