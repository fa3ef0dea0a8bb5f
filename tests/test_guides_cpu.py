"""CPU tests of the guide buffers' host-visible surface: the ctypes prototype of rayz_cuda_render_guides against
include/rayz_cuda.h and the Zig externs, loud failures (never a fallback) without a context or a device, and the C++ host's PFM
writer (host/rayz_host.hpp writePFM, the format of rayz_host --guides): header, bottom-up rows and exact float bytes."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

from rayz_b200 import _abi as abi

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


def test_ctypes_prototype_matches_header():
    hdr = open(os.path.join(ROOT, "include", "rayz_cuda.h")).read()
    proto = re.search(r"int rayz_cuda_render_guides\(([^)]*)\);", hdr)
    assert proto and [a.strip() for a in proto.group(1).split(",")] == [
        "RzContext *ctx", "const RzCamera *cam", "const RzRenderParams *p", "float *out_albedo", "float *out_normal"]
    res, args = abi.SYMBOLS["rayz_cuda_render_guides"]
    assert res is C.c_int and args == [C.c_void_p, C.POINTER(abi.RzCamera), C.POINTER(abi.RzRenderParams), C.c_void_p, C.c_void_p]
    assert re.search(r"#define RAYZ_CUDA_ABI_VERSION 3\b", hdr)
    lib = abi.load()
    assert lib.rayz_cuda_abi_version() == 3
    zig = open(os.path.join(ROOT, "zig", "cuda_backend.zig")).read()
    assert "pub extern fn rayz_cuda_render_guides(ctx: *RzContext, cam: *const RzCamera, params: *const RzRenderParams, " \
           "out_albedo: ?[*]f32, out_normal: ?[*]f32) c_int;" in zig


def test_render_guides_fails_loudly_without_a_context():
    lib = abi.load()
    p = abi.RzRenderParams()
    p.width, p.height, p.spp = 8, 8, 4
    cam = abi.RzCamera()
    out = np.zeros(8 * 8 * 4, dtype=np.float32)
    assert lib.rayz_cuda_render_guides(None, C.byref(cam), C.byref(p), out.ctypes.data, out.ctypes.data) == -1
    assert lib.rayz_cuda_last_error().startswith(b"guides:") and b"NULL" in lib.rayz_cuda_last_error()
    assert (out == 0).all()


def test_no_gpu_means_no_guides_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    import rayz_b200
    t = rayz_b200.random_bouncing(32, seed=42)
    with pytest.raises(abi.BackendError) as e:
        t.render_guides()
    assert e.value.code == -2 and "no CPU path" in str(e.value)
    assert t.albedo is None and t.normal is None


@pytest.fixture(scope="module")
def pfm_check():
    exe = os.path.join(HERE, "_build", "pfm_check")
    src = os.path.join(HERE, "hostsim", "pfm_check.cpp")
    hdr = os.path.join(ROOT, "host", "rayz_host.hpp")
    os.makedirs(os.path.dirname(exe), exist_ok=True)
    if not os.path.exists(exe) or os.path.getmtime(exe) < max(os.path.getmtime(src), os.path.getmtime(hdr)):
        subprocess.run(["g++", "-O2", "-std=c++17", "-o", exe, src], check=True)
    return exe


def lcg_floats(n: int, seed: int) -> np.ndarray:
    out = np.empty(n, dtype=np.float32)
    s = seed
    for i in range(n):
        s = (s * 6364136223846793005 + 1442695040888963407) & 0xFFFFFFFFFFFFFFFF
        out[i] = ((s >> 40) - (1 << 23)) / (1 << 20)
    return out


@pytest.mark.parametrize("w,h", [(1, 1), (7, 3), (5, 11)])
def test_pfm_writer_layout(pfm_check, tmp_path, w, h):
    prefix = str(tmp_path / "g")
    r = subprocess.run([pfm_check, str(w), str(h), "7", prefix], capture_output=True, text=True, check=True)
    px = lcg_floats(w * h * 4, 7).reshape(h, w, 4)
    for suffix, tag, chans in (("_rgb.pfm", b"PF", px[..., :3]), ("_w.pfm", b"Pf", px[..., 3])):
        got = open(prefix + suffix, "rb").read()
        head = tag + f"\n{w} {h}\n-1.0\n".encode()
        assert got[:len(head)] == head
        body = np.ascontiguousarray(chans[::-1], dtype="<f4").tobytes()   # the bottom row first, little-endian
        assert got[len(head):] == body
    assert [int(x) for x in r.stdout.split()] == [os.path.getsize(prefix + "_rgb.pfm"), os.path.getsize(prefix + "_w.pfm")]
