#!/bin/bash
# Test-only: compiles the pooled adaptive estimate (rz_device.cuh's RZ_RENDER_ADAPTIVE_POOLED pieces) as host code (see pooled.cu).
set -e
cd "$(dirname "$0")"
mkdir -p ../_build
SO=../_build/libhostpool.so
if [ ! -f $SO ] || [ pooled.cu -nt $SO ] || [ ../../rayz_b200/csrc/rz_sampler.cuh -nt $SO ] || [ ../../rayz_b200/csrc/rz_device.cuh -nt $SO ]; then
  nvcc -x cu -O2 -std=c++17 -shared -Xcompiler -fPIC -Wno-deprecated-gpu-targets -o $SO pooled.cu
fi
