#!/bin/bash
# Builds occupancy/capacity variants of librayz_cuda.so that differ in the numeric compile-time constants of ONE source file
# (RZ_PRIMARY_MINB, RZ_SECOND_MINB of rz_path.cu; RZ_BVH_MINB, RZ_BVH_CAMERA_MINB, RZ_CL_CAP, RZ_CL_WL with SRC=rz_bvh_trace.cu),
# as scripts/_build/exp/<name>.so; scripts/exp_probe.py / exp_bvh.py --so load one of them instead of the product library.
#   [SRC=rz_bvh_trace.cu] scripts/exp_build.sh name1 "-DFLAG=1 ..." [name2 "flags" ...]
set -e
cd "$(dirname "$0")/.."
python -m rayz_b200.build > /dev/null
mkdir -p scripts/_build/exp
[ -n "$KEEP" ] || rm -f scripts/_build/exp/*.so
OBJ=rayz_b200/lib/obj
SRC=${SRC:-rz_path.cu}
build() {   # name, flags...
  local name=$1; shift
  nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -lineinfo -Xcompiler -fPIC -Xcompiler -fvisibility=default --use_fast_math $@ \
       -c rayz_b200/csrc/$SRC -o scripts/_build/exp/$name.o
  local objs=""; for o in $OBJ/*.o; do [ "$(basename $o)" = "${SRC%.cu}.o" ] || objs="$objs $o"; done
  nvcc -gencode arch=compute_100a,code=sm_100a -shared -o scripts/_build/exp/$name.so scripts/_build/exp/$name.o $objs -cudart static -Xlinker --no-undefined
  rm -f scripts/_build/exp/$name.o
}
while [ $# -ge 2 ]; do build "$1" $2 & shift 2; done
wait
ls -la scripts/_build/exp
