#!/bin/bash
# Test-only: compiles the light-path pass rule (rz_device.cuh's RZ_RENDER_PASSES pieces) as host code (see passes.cu).
set -e
cd "$(dirname "$0")"
mkdir -p ../_build
SO=../_build/libhostpass.so
if [ ! -f $SO ] || [ passes.cu -nt $SO ] || [ ../../rayz_b200/csrc/rz_sampler.cuh -nt $SO ] || [ ../../rayz_b200/csrc/rz_device.cuh -nt $SO ] || [ ../../include/rayz_cuda.h -nt $SO ]; then
  nvcc -x cu -O2 -std=c++17 -shared -Xcompiler -fPIC -Wno-deprecated-gpu-targets -o $SO passes.cu
fi
