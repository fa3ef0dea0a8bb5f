#!/bin/bash
# Test-only: compiles the pixel filters' warp and the camera-stage culls (rz_device.cuh) as host code (see filter.cu).
set -e
cd "$(dirname "$0")"
mkdir -p ../_build
SO=../_build/libhostfilter.so
if [ ! -f $SO ] || [ filter.cu -nt $SO ] || [ ../../rayz_b200/csrc/rz_sampler.cuh -nt $SO ] || [ ../../rayz_b200/csrc/rz_device.cuh -nt $SO ] || [ ../../rayz_b200/csrc/rz_filter_table.h -nt $SO ] || [ ../../include/rayz_cuda.h -nt $SO ]; then
  nvcc -x cu -O2 -std=c++17 -shared -Xcompiler -fPIC -Xcompiler -pthread -Wno-deprecated-gpu-targets -o $SO filter.cu
fi
