#!/bin/bash
# Test-only: compiles the denoiser's arithmetic (rz_denoise.cuh) on its own as host code (see denoise.cu).
set -e
cd "$(dirname "$0")"
mkdir -p ../_build
SO=../_build/libhostdenoise.so
if [ ! -f $SO ] || [ denoise.cu -nt $SO ] || [ ../../rayz_b200/csrc/rz_denoise.cuh -nt $SO ] || [ ../../rayz_b200/csrc/rz_device.cuh -nt $SO ]; then
  nvcc -x cu -O2 -std=c++17 -shared -Xcompiler -fPIC -Wno-deprecated-gpu-targets -o $SO denoise.cu
fi
