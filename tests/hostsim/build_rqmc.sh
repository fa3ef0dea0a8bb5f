#!/bin/bash
# Test-only: compiles the randomised-QMC estimate (rz_sampler.cuh's replicates, rz_device.cuh's segment gain) as host code (see rqmc.cu).
set -e
cd "$(dirname "$0")"
mkdir -p ../_build
SO=../_build/libhostrqmc.so
if [ ! -f $SO ] || [ rqmc.cu -nt $SO ] || [ ../../rayz_b200/csrc/rz_sampler.cuh -nt $SO ] || [ ../../rayz_b200/csrc/rz_device.cuh -nt $SO ]; then
  nvcc -x cu -O2 -std=c++17 -shared -Xcompiler -fPIC -Wno-deprecated-gpu-targets -o $SO rqmc.cu
fi
