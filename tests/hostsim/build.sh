#!/bin/bash
# Test-only: compiles the product's FP32 device shading header as HOST code (see hostsim.cu).
set -e
cd "$(dirname "$0")"
mkdir -p ../_build
if [ ! -f ../_build/libhostsim.so ] || [ hostsim.cu -nt ../_build/libhostsim.so ] || [ ../../rayz_b200/csrc/rz_device.cuh -nt ../_build/libhostsim.so ] || [ ../../rayz_b200/csrc/rz_sampler.cuh -nt ../_build/libhostsim.so ] || [ ../../rayz_b200/csrc/rz_host_bvh.hpp -nt ../_build/libhostsim.so ] || [ ../../rayz_b200/csrc/rz_launch.h -nt ../_build/libhostsim.so ]; then  # rebuilt whenever the header changes
  nvcc -x cu -O2 -std=c++17 -shared -Xcompiler -fPIC,-pthread -Wno-deprecated-gpu-targets -o ../_build/libhostsim.so hostsim.cu
fi
