#!/bin/bash
# Test-only: compiles the low-discrepancy sampler (rz_sampler.cuh) as host code (see sampler.cu).
set -e
cd "$(dirname "$0")"
mkdir -p ../_build
SO=../_build/libhostsampler.so
if [ ! -f $SO ] || [ sampler.cu -nt $SO ] || [ ../../rayz_b200/csrc/rz_sampler.cuh -nt $SO ] || [ ../../rayz_b200/csrc/rz_device.cuh -nt $SO ]; then
  nvcc -x cu -O2 -std=c++17 -shared -Xcompiler -fPIC -Wno-deprecated-gpu-targets -o $SO sampler.cu
fi
