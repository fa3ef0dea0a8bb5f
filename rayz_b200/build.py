"""Builds librayz_cuda.so (the C-ABI CUDA backend) in-tree for sm_100a with nvcc.

    python -m rayz_b200.build [--force]

nvcc cross-compiles without a GPU.  The .so lands in rayz_b200/lib/ (git-ignored, shipped to the
GPU box by gpurun).  rz_ids.cu is compiled with --fmad=false (bit-exact f64, see the file header);
the FP32 path kernels with --use_fast_math (FTZ, approximate sqrt/rsqrt in the search loop; the
winning hit is re-evaluated in f64).
"""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
OBJDIR = os.path.join(LIBDIR, "obj")
SO = os.path.join(LIBDIR, "librayz_cuda.so")
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=default"]
UNITS = {
    "rz_path.cu": ["--use_fast_math"],
    "rz_wavefront.cu": ["--use_fast_math"],
    "rz_misc.cu": [],
    "rz_denoise.cu": [],
    "rz_adaptive.cu": [],
    "rz_ids.cu": ["--fmad=false"],
    "rz_bvh_build.cu": [],
    "rz_sort.cu": [],
    "rz_bvh_trace.cu": ["--use_fast_math"],
    "rz_context.cu": [],
}
HEADERS = ["rz_device.cuh", "rz_sampler.cuh", "rz_search.cuh", "rz_denoise.cuh", "rz_launch.h", os.path.join("..", "..", "include", "rayz_cuda.h")]


def _nvcc() -> str:
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if c and (os.path.isabs(c) and os.path.exists(c) or not os.path.isabs(c)):
            return c
    raise RuntimeError("nvcc not found")


def _stale(target: str, deps) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(OBJDIR, exist_ok=True)
    nvcc = _nvcc()
    hdrs = [os.path.join(CSRC, h) for h in HEADERS] + [os.path.abspath(__file__)]
    jobs = []
    objs = []
    for src, extra in UNITS.items():
        s = os.path.join(CSRC, src)
        o = os.path.join(OBJDIR, src.replace(".cu", ".o"))
        objs.append(o)
        if force or _stale(o, [s] + hdrs):
            jobs.append([nvcc] + ARCH + COMMON + extra + (["-Xptxas", "-v"] if verbose else []) + ["-c", s, "-o", o])

    def run(cmd):
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + r.stdout + r.stderr)
        return r.stderr

    with ThreadPoolExecutor(max_workers=min(8, max(1, len(jobs)))) as ex:
        for out in ex.map(run, jobs):
            if verbose and out:
                print(out)
    if force or jobs or _stale(SO, objs):
        run([nvcc] + ARCH + ["-shared", "-o", SO] + objs + ["-cudart", "static", "-Xlinker", "--no-undefined"])
    return SO


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
