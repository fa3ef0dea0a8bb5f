"""CPU tests of adaptive sampling's host-visible surface: the ctypes mirror of RZ_RENDER_ADAPTIVE and rayz_cuda_pixel_samples
against include/rayz_cuda.h, and loud failures (never a fallback) without a context or a device."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from rayz_b200 import _abi as abi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_ctypes_mirror_matches_header():
    hdr = open(os.path.join(ROOT, "include", "rayz_cuda.h")).read()
    m = re.search(r"#define RZ_RENDER_ADAPTIVE\s+(0x[0-9a-fA-F]+|\d+)u", hdr)
    assert m and int(m.group(1), 0) == abi.RENDER_ADAPTIVE == 8
    # a bit of its own
    assert abi.RENDER_ADAPTIVE & (abi.RENDER_SERIAL_PASSES | abi.RENDER_MOMENTS | abi.RENDER_ACCUMULATE) == 0
    proto = re.search(r"int rayz_cuda_pixel_samples\(([^)]*)\);", hdr)
    assert proto and [a.strip() for a in proto.group(1).split(",")] == ["RzContext *ctx", "uint32_t *out_spp"]
    res, args = abi.SYMBOLS["rayz_cuda_pixel_samples"]
    assert res is C.c_int and args == [C.c_void_p, C.c_void_p]
    lib = abi.load()
    assert lib.rayz_cuda_abi_version() == 3
    zig = open(os.path.join(ROOT, "zig", "cuda_backend.zig")).read()
    assert "pub const RZ_RENDER_ADAPTIVE: u32 = 8;" in zig and "pub extern fn rayz_cuda_pixel_samples(" in zig


def test_new_calls_fail_loudly_without_a_context():
    lib = abi.load()
    out = np.zeros(16, dtype=np.uint32)
    assert lib.rayz_cuda_pixel_samples(None, out.ctypes.data) == -1
    assert b"NULL" in lib.rayz_cuda_last_error()
    p = abi.RzRenderParams()
    p.width, p.height, p.spp, p.flags = 8, 8, 4, abi.RENDER_ADAPTIVE
    cam, nz = abi.RzCamera(), abi.RzNoise()
    assert lib.rayz_cuda_render_to_noise(None, C.byref(cam), C.byref(p), 0.01, 64, None, None, None, C.byref(nz)) == -1
    assert b"NULL" in lib.rayz_cuda_last_error()
    # the plain render calls refuse the bit before they look at anything else
    assert lib.rayz_cuda_render(None, C.byref(cam), C.byref(p), None, None, None) == -1
    assert b"RZ_RENDER_ADAPTIVE" in lib.rayz_cuda_last_error()
    assert lib.rayz_cuda_render_device(None, C.byref(cam), C.byref(p), None, None, None, 1) == -1
    assert b"RZ_RENDER_ADAPTIVE" in lib.rayz_cuda_last_error()


def test_no_gpu_means_no_adaptive_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    import rayz_b200
    t = rayz_b200.random_bouncing(32, seed=42)
    with pytest.raises(abi.BackendError) as e:
        t.render(noise_target=2 / 255, max_spp=64, adaptive=True)
    assert e.value.code == -2 and "no CPU path" in str(e.value)
    assert t.pixel_samples is None
    with pytest.raises(abi.BackendError) as e:
        rayz_b200.Backend((0,))
    assert e.value.code == -2
