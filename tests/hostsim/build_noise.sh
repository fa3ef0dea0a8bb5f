#!/bin/bash
# Test-only: compiles the noise estimate of progressive rendering (rz_device.cuh) on its own as host code (see noise.cu).
set -e
cd "$(dirname "$0")"
mkdir -p ../_build
SO=../_build/libhostnoise.so
if [ ! -f $SO ] || [ noise.cu -nt $SO ] || [ ../../rayz_b200/csrc/rz_device.cuh -nt $SO ]; then
  nvcc -x cu -O2 -std=c++17 -shared -Xcompiler -fPIC -Wno-deprecated-gpu-targets -o $SO noise.cu
fi
