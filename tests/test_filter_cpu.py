"""CPU tests of the pixel filters (include/rayz_cuda.h "RZ_RENDER_FILTER"): the warp the kernels run, compiled as host code
(tests/hostsim/filter.cu), over every one of the 2^24 jitter uniforms against the f64 CDF (filter_replay.py); the Sobol
strata it keeps; the two camera-stage culls with a filter's footprint; the f64 restatement of filtered camera rays the GPU
tests use; and the field's declarations in every layer."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

import rayz_b200
from rayz_b200 import Backend
from rayz_b200 import _abi as abi
import filter_replay as fr
import mattes_replay

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = open(os.path.join(ROOT, "include", "rayz_cuda.h")).read()
ZIG = open(os.path.join(ROOT, "zig", "cuda_backend.zig")).read()
KINDS = [fr.TENT, fr.GAUSSIAN, fr.BLACKMAN_HARRIS]
ALL_U = np.arange(1 << 24, dtype=np.float32) * np.float32(2.0 ** -24)   # every 24-bit jitter uniform (rz_u01)


@pytest.fixture(scope="module")
def lib():
    subprocess.run(["bash", os.path.join(ROOT, "tests", "hostsim", "build_filter.sh")], check=True)
    L = C.CDLL(os.path.join(ROOT, "tests", "_build", "libhostfilter.so"))
    L.hostfilt_warp.argtypes = [C.c_uint32, C.c_uint32, C.c_void_p, C.c_uint64, C.c_void_p, C.c_int]
    L.hostfilt_width16.argtypes = [C.c_uint32]
    L.hostfilt_width16.restype = C.c_uint32
    L.hostfilt_reach.argtypes = [C.c_uint32]
    L.hostfilt_reach.restype = C.c_float
    L.hostfilt_sobol_jitter.argtypes = [C.c_uint32] * 5 + [C.c_int, C.c_uint32] + [C.c_void_p] * 4
    L.hostfilt_lens_ray.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p]
    L.hostfilt_cull_check.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_int, C.c_uint32, C.c_float, C.c_uint64, C.c_uint64,
                                      C.c_void_p]
    return L


def warp(lib, kind, width16, u):
    u = np.ascontiguousarray(u, np.float32)
    out = np.empty_like(u)
    lib.hostfilt_warp(kind, width16, u.ctypes.data, len(u), out.ctypes.data, os.cpu_count() or 1)
    return out


# ------------------------------------------------------------------------------- 1. the warp, at every uniform
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("width", [1.0, None, 4.0])
def test_warp_at_every_uniform(lib, kind, width):
    """Monotone, inside [-R, R], odd about 1/2, within 1e-5 px of the exact inverse CDF and |F(w(u)) - u| <= 2^-21, at each of
    the 2^24 uniforms the samplers draw.  The 1e-5 px bound is checked exactly, without a bisection per uniform: F is
    increasing, so |w(u) - w*(u)| <= e iff F(w(u) - e) <= u <= F(w(u) + e)."""
    W = fr.DEFAULT_WIDTH[kind] if width is None else width
    x = warp(lib, kind, int(W * 16), ALL_U)   # rz_filter_warp takes the width resolved (rz_filter_width16)
    R = W / 2
    assert np.all(np.diff(x) >= 0), "not monotone"
    assert x.min() >= -R and x.max() <= R
    assert x[0] == -R, "u = 0 starts at the support's edge"
    # odd about 1/2: w(1 - u) = -w(u) (1 - u is exact for every 24-bit u)
    assert np.max(np.abs(x[1:][::-1].astype(np.float64) + x[1:])) <= 1e-6
    assert x[1 << 23] == 0.0
    u64, x64 = ALL_U.astype(np.float64), x.astype(np.float64)
    F = fr.cdf(kind, W, x64)
    ks = np.max(np.abs(F - u64))
    e = 1e-5
    lo_ok = fr.cdf(kind, W, x64 - e) <= u64
    hi_ok = fr.cdf(kind, W, x64 + e) >= u64
    print(f"kind {kind} width {W}: max |F(w(u)) - u| = {ks:.3g} (2^-21 = {2.0 ** -21:.3g})")
    assert ks <= 2.0 ** -21
    assert lo_ok.all() and hi_ok.all(), f"{int((~lo_ok | ~hi_ok).sum())} uniforms more than 1e-5 px from the exact warp"


@pytest.mark.parametrize("kind", KINDS)
def test_warp_against_the_bisection_reference(lib, kind):
    """Against filter_replay.filter_warp (bisection on the f64 CDF) directly, tails included: the first and last 2^12
    uniforms and a stride through the rest, at the widest width."""
    idx = np.unique(np.concatenate([np.arange(4096), np.arange(0, 1 << 24, 997), (1 << 24) - 1 - np.arange(4096)]))
    u = ALL_U[idx]
    x = warp(lib, kind, 64, u).astype(np.float64)
    ref = fr.filter_warp(kind, 4.0, u.astype(np.float64))
    worst = np.max(np.abs(x - ref))
    print(f"kind {kind}: max |w - w*| = {worst:.3g} px over {len(u)} uniforms")
    assert worst <= 1e-5


def test_box_is_the_reference_jitter_bit_for_bit(lib):
    assert np.array_equal(warp(lib, fr.BOX, 0, ALL_U).view(np.uint32), (ALL_U - np.float32(0.5)).view(np.uint32))


def test_width_field_defaults_and_reach(lib):
    for kind, w16 in ((fr.BOX, 16), (fr.TENT, 32), (fr.GAUSSIAN, 48), (fr.BLACKMAN_HARRIS, 24)):
        assert lib.hostfilt_width16(abi.render_filter(kind)) == w16
        assert lib.hostfilt_width16(abi.render_filter(kind, 40)) == 40
    assert lib.hostfilt_reach(abi.render_filter(fr.BOX)) == 0.5
    assert lib.hostfilt_reach(abi.render_filter(fr.BLACKMAN_HARRIS, 16)) == 0.5     # a 1 px filter reaches no further than the box
    assert lib.hostfilt_reach(abi.render_filter(fr.GAUSSIAN)) == 1.5
    assert lib.hostfilt_reach(abi.render_filter(fr.TENT, 64)) == 2.0


# ------------------------------------------------------------------------------- 2. Sobol strata
@pytest.mark.parametrize("kind,w16", [(fr.TENT, 0), (fr.GAUSSIAN, 64), (fr.BLACKMAN_HARRIS, 0)])
@pytest.mark.parametrize("rqmc", [False, True])
def test_sobol_strata_map_to_equal_filter_mass(lib, kind, w16, rqmc):
    """Aligned blocks of 2^k samples of a pixel's camera-jitter pair are (0, k, 2)-nets: one point per 2^-a x 2^-b box.  The
    warp is monotone per axis, so the warped points fall one per box of the filter's quantile grid (boundaries w(j 2^-a)),
    and those boundaries are the exact quantiles to 1e-5 px."""
    flags = abi.render_filter(kind, w16)
    w16 = lib.hostfilt_width16(flags)
    W = w16 / 16
    for gpix, s0 in ((0, 0), (12345, 1024), (777777, 3 * 1024)):
        n = 1024
        ux, uy, wx, wy = (np.empty(n, np.float32) for _ in range(4))
        lib.hostfilt_sobol_jitter(0x1234, 0x5678, gpix, s0, n, int(rqmc), flags, *(a.ctypes.data for a in (ux, uy, wx, wy)))
        # under RQMC a pixel's samples alternate between two replicates: each replicate's own sequence is the net
        streams = [slice(0, None, 2), slice(1, None, 2)] if rqmc else [slice(None)]
        for sl in streams:
            px, py = wx[sl], wy[sl]
            for k in range(0, 10 if rqmc else 11):
                for a in range(k + 1):
                    b = k - a
                    qa = warp(lib, kind, w16, (np.arange(1, 1 << a) * 2.0 ** -a).astype(np.float32))
                    qb = warp(lib, kind, w16, (np.arange(1, 1 << b) * 2.0 ** -b).astype(np.float32))
                    for blk in range(0, len(px), 1 << k):
                        ix = np.searchsorted(qa, px[blk:blk + (1 << k)], side="right")
                        iy = np.searchsorted(qb, py[blk:blk + (1 << k)], side="right")
                        cells = ix * (1 << b) + iy
                        assert len(np.unique(cells)) == 1 << k, (gpix, s0, k, a, blk)
    q = warp(lib, kind, w16, (np.arange(1, 1024) / 1024).astype(np.float32)).astype(np.float64)
    assert np.max(np.abs(q - fr.filter_warp(kind, W, np.arange(1, 1024) / 1024))) <= 1e-5


# ------------------------------------------------------------------------------- 3. the culls widen to the support
def _cam(width, defocus_angle, look_from=(13, 2, 3), vfov=20.0):
    h = int(width / rayz_b200.host.ASPECT_RATIO)
    return rayz_b200.Camera.init(vfov, 10.0, defocus_angle, look_from, (0, 0, 0), (0, 1, 0), h, width).rz, h


@pytest.mark.parametrize("flags", [abi.render_filter(abi.FILTER_GAUSSIAN, 64), abi.render_filter(abi.FILTER_TENT),
                                   abi.render_filter(abi.FILTER_BLACKMAN_HARRIS), abi.render_filter(abi.FILTER_TENT, 64)])
@pytest.mark.parametrize("width,defocus,look_from,vfov", [
    (1200, 0.6, (13, 2, 3), 20.0),        # the benchmark camera
    (400, 0.0, (13, 2, 3), 20.0),         # pinhole
    (160, 8.0, (0, 1.0, 8.0), 50.0),      # wide lens, wide field, coarse pixels
    (33, 2.0, (3, 3, 2), 90.0),           # tiles that wrap around image rows
])
@pytest.mark.parametrize("block", [0, 1])
def test_camera_stage_culls_never_drop_a_hit_sphere_under_a_filter(lib, flags, width, defocus, look_from, vfov, block):
    """The staged K1's 32-pixel tile cone (block = 0) and K3's 8 x 4 block cone (block = 1, boxes too) with the corners at
    +-max(0.5, R): every sphere a filtered camera ray hits is kept, for rays whose offsets reach +-R exactly."""
    cam, h = _cam(width, defocus, look_from, vfov)
    out = np.zeros(5, dtype=np.uint64)
    assert lib.hostfilt_cull_check(C.addressof(cam), width, h, block, flags, 0.0, 2500, 11, out.ctypes.data) == 0
    dropped, hits, boxes_dropped, boxes, culled = (int(x) for x in out)
    assert hits > 100_000
    assert dropped == 0, f"{dropped} of {hits} hit spheres culled"
    assert boxes_dropped == 0, f"{boxes_dropped} of {boxes} boxes around hit spheres culled"
    if width >= 400:
        assert culled > 1_000


@pytest.mark.parametrize("block", [0, 1])
def test_the_pixel_footprint_alone_drops_filtered_hits(lib, block):
    """The check above tells: with the box's cone (corners at +-0.5 px) the rays of a 4 px Gaussian lose hit spheres."""
    cam, h = _cam(400, 0.0)
    out = np.zeros(5, dtype=np.uint64)
    lib.hostfilt_cull_check(C.addressof(cam), 400, h, block, abi.render_filter(abi.FILTER_GAUSSIAN, 64), 0.5, 2500, 11,
                            out.ctypes.data)
    assert int(out[0]) > 0


# ------------------------------------------------------------------------------- 4. the f64 restatement of filtered rays
def test_box_camera_rays_equal_the_matte_replays():
    arrays, cam = None, rayz_b200.Camera.init(20.0, 10.0, 0.6, (13, 2, 3), (0, 0, 0), (0, 1, 0), 9, 16).rz
    for sampler in ("philox", "sobol"):
        a = fr.camera_rays(cam, 16, 9, 3, 2, 11, sampler)
        b = mattes_replay.camera_rays(cam, 16, 9, 3, 2, 11, sampler)
        for x, y in zip(a, b):
            assert np.array_equal(x, y)


@pytest.mark.parametrize("pixel_filter,filter_width", [("tent", None), ("gaussian", 4.0), ("blackman-harris", None)])
@pytest.mark.parametrize("defocus", [0.0, 0.6])
def test_filtered_camera_rays_equal_the_kernels_rays(lib, pixel_filter, filter_width, defocus):
    """Each restated camera ray is getRay at the warped position: the host-compiled rz_lens_ray over the same uniforms agrees
    to f32 rounding."""
    import oracle
    w, h, spp, seed = 24, 13, 3, 11
    cam = rayz_b200.Camera.init(20.0, 10.0, defocus, (13, 2, 3), (0, 0, 0), (0, 1, 0), h, w).rz
    o, d, t = fr.camera_rays(cam, w, h, 5, spp, seed, "philox", pixel_filter, filter_width)
    flags = fr.flags_of(pixel_filter, filter_width)
    worst = 0.0
    for j in range(h):
        for i in range(w):
            for s in range(spp):
                u5 = np.ascontiguousarray(oracle.replay_uniforms(seed, j * w + i, 5 + s, 0)[:5], np.float32)
                od = np.empty(6, np.float32)
                lib.hostfilt_lens_ray(C.addressof(cam), i, j, u5.ctypes.data, flags, od.ctypes.data)
                worst = max(worst, np.abs(od[3:] - d[j, i, s]).max())
                assert np.abs(od[:3] - o[j, i, s]).max() < 1e-5
    assert worst < 2e-6, worst


# ------------------------------------------------------------------------------- 5. the field in every layer
def test_constants_in_every_layer():
    for name, value in (("RZ_RENDER_FILTER_SHIFT", 8), ("RZ_RENDER_FILTER_MASK", 0x300), ("RZ_RENDER_FILTER_WIDTH_SHIFT", 16),
                        ("RZ_RENDER_FILTER_WIDTH_MASK", 0xFF0000), ("RZ_FILTER_BOX", 0), ("RZ_FILTER_TENT", 1),
                        ("RZ_FILTER_GAUSSIAN", 2), ("RZ_FILTER_BLACKMAN_HARRIS", 3), ("RZ_FILTER_WIDTH_MIN", 16),
                        ("RZ_FILTER_WIDTH_MAX", 64)):
        m = re.search(rf"#define {name} (0x[0-9a-fA-F]+|\d+)u?\b", HEADER)
        assert m and int(m.group(1), 0) == value, name
        assert getattr(abi, name[3:]) == value, name
        z = re.search(rf"pub const {name}\b[^=]*= (0x[0-9a-fA-F]+|\d+);", ZIG)
        assert z and int(z.group(1), 0) == value, name
    assert "RZ_RENDER_FILTER(kind, width16)" in HEADER


def test_backend_params_encode_the_filter():
    assert Backend.params(8, 8, 1).flags & (abi.RENDER_FILTER_MASK | abi.RENDER_FILTER_WIDTH_MASK) == 0
    p = Backend.params(8, 8, 1, pixel_filter="gaussian", filter_width=3.5, sobol=True)
    assert p.flags == abi.RENDER_SOBOL | (2 << 8) | (56 << 16)
    assert Backend.params(8, 8, 1, pixel_filter="blackman-harris").flags == 3 << 8
    with pytest.raises(ValueError):
        Backend.params(8, 8, 1, pixel_filter="mitchell")
    with pytest.raises(ValueError):
        Backend.params(8, 8, 1, pixel_filter="tent", filter_width=1.03)
    t = rayz_b200.Tracer.__new__(rayz_b200.Tracer)
    t.sampler, t.pixel_filter, t.filter_width = "sobol", "tent", 2.5
    assert t._sampler() == {"sobol": True} and t._filter() == {"pixel_filter": "tent", "filter_width": 2.5}
