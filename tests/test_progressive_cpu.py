"""CPU tests of progressive rendering's host-visible parts: the per-pixel noise estimate (rz_device.cuh's rz_pixel_err and the
fixed-point quantisation of the kernels' sky branch, compiled as host code by tests/hostsim/noise.cu) against numpy f64, and the
ctypes mirror of the new C-ABI surface."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

from rayz_b200 import _abi as abi

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
FLOOR = 1e-4   # RZ_NOISE_Y_FLOOR


@pytest.fixture(scope="module")
def hs():
    subprocess.run(["bash", os.path.join(HERE, "hostsim", "build_noise.sh")], check=True)
    lib = C.CDLL(os.path.join(HERE, "_build", "libhostnoise.so"))
    lib.hostnoise_moments.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p]
    lib.hostnoise_pixel_err.argtypes = [C.c_void_p, C.c_uint32]
    lib.hostnoise_pixel_err.restype = C.c_double
    return lib


def quantise(hs, rgb):
    """Per-path radiances [n, 3] -> the pixel's four accumulator slots, as the kernels add them."""
    rgb = np.ascontiguousarray(rgb, dtype=np.float32)
    q = np.zeros(4, dtype=np.uint64)
    hs.hostnoise_moments(rgb.ctypes.data, rgb.shape[0], q.ctypes.data)
    return q


def err_gpu_formula(hs, q, n):
    q = np.ascontiguousarray(q, dtype=np.uint64)
    return hs.hostnoise_pixel_err(q.ctypes.data, n)


def err_numpy(q, n):
    """The formula of include/rayz_cuda.h (rayz_cuda_noise) in numpy f64."""
    if n < 2:
        return np.inf
    s = 2.0 ** -32
    q = [float(int(x)) for x in q]
    y = (0.2126 * q[0] + 0.7152 * q[1] + 0.0722 * q[2]) * s / n
    s2 = max(0.0, q[3] * s / n - y * y) * n / (n - 1)
    return np.sqrt(s2 / n) / (2.0 * np.sqrt(max(y, FLOOR)))


def err_from_samples(rgb):
    """Textbook estimate from the unquantised samples: standard error of the mean luminance, through the gamma-2 slope."""
    rgb = np.clip(np.asarray(rgb, dtype=np.float64), 0, 2.0 ** 20)
    y = rgb @ np.array([0.2126, 0.7152, 0.0722])
    n = y.size
    return np.sqrt(y.var(ddof=1) / n) / (2.0 * np.sqrt(max(y.mean(), FLOOR)))


def test_quantisation_matches_numpy(hs):
    rng = np.random.default_rng(1)
    rgb = rng.uniform(0, 1.5, (1000, 3)).astype(np.float32)
    rgb[::7] = 0
    rgb[3] = (-1.0, 2.0e6, 0.5)   # clamped to [0, 2^20] like the colour atomics
    q = quantise(hs, rgb)
    c = np.clip(rgb, 0, np.float32(2.0 ** 20))
    want = [int(np.sum(np.rint(c[:, k].astype(np.float64) * 2.0 ** 32))) for k in range(3)]
    assert [int(x) for x in q[:3]] == want
    y = np.float32(0.0722) * c[:, 2] + (np.float32(0.7152) * c[:, 1] + np.float32(0.2126) * c[:, 0])
    y2 = np.clip(y.astype(np.float64) ** 2, 0, 2.0 ** 20)
    # the product rounds y in FP32 with explicit FMAs: the sum of squares agrees to FP32 rounding of each term
    assert abs(int(q[3]) - np.sum(y2 * 2.0 ** 32)) <= 1e-6 * np.sum(y2 * 2.0 ** 32)


@pytest.mark.parametrize("case", ["uniform", "sky_or_black", "bright", "large_n"])
def test_pixel_err_matches_numpy(hs, case):
    rng = np.random.default_rng(["uniform", "sky_or_black", "bright", "large_n"].index(case) + 10)
    if case == "uniform":
        rgb = rng.uniform(0, 1, (64, 3))
    elif case == "sky_or_black":   # a path either reaches the sky or is absorbed: the typical pixel
        rgb = np.where(rng.uniform(size=(256, 1)) < 0.3, rng.uniform(0.3, 1.0, (256, 3)), 0.0)
    elif case == "bright":
        rgb = rng.uniform(50, 60, (32, 3))
    else:
        rgb = rng.uniform(0, 1, (200_000, 3)) ** 3
    n = rgb.shape[0]
    q = quantise(hs, rgb)
    got = err_gpu_formula(hs, q, n)
    assert got == pytest.approx(err_numpy(q, n), rel=1e-12, abs=1e-15)
    # and it is the textbook standard error of the displayed value, up to FP32 luminance and 2^-32 quantisation
    assert got == pytest.approx(err_from_samples(rgb.astype(np.float32)), rel=1e-4)


def test_constant_samples_give_zero(hs):
    for v in ((0.5, 0.5, 0.5), (0.25, 0.75, 1.0), (0.0, 0.0, 0.0), (3.0, 2.0, 1.0)):
        for n in (2, 17, 4096):
            q = quantise(hs, np.tile(np.array(v, dtype=np.float32), (n, 1)))
            e = err_gpu_formula(hs, q, n)
            # zero up to the FP32 rounding of each path's Y (a relative 2^-24 that Ybar, taken from the f64 sums of the three
            # channels, does not share): sigma <= Ybar sqrt(2^-22 / (n - 1)), a small fraction of one 8-bit step even at n = 2
            ybar = 0.2126 * v[0] + 0.7152 * v[1] + 0.0722 * v[2]
            assert 0.0 <= e <= ybar * np.sqrt(2.0 ** -22 / (n - 1)) / (2 * np.sqrt(max(ybar, FLOOR))) + 1e-15, (v, n, e)
            if n >= 17:
                assert e < 0.05 / 255
            assert e == pytest.approx(err_numpy(q, n), abs=1e-15)


def test_one_sample_has_no_estimate(hs):
    q = quantise(hs, np.array([[0.3, 0.4, 0.5]], dtype=np.float32))
    assert np.isinf(err_gpu_formula(hs, q, 1)) and err_gpu_formula(hs, q, 1) > 0
    assert np.isinf(err_gpu_formula(hs, np.zeros(4, np.uint64), 0))


def test_black_pixels_hit_the_floor(hs):
    # a dark pixel: one path in 1000 carries a little light; its mean luminance is far below the floor
    n = 1000
    rgb = np.zeros((n, 3), dtype=np.float32)
    rgb[17] = (0.02, 0.02, 0.02)
    q = quantise(hs, rgb)
    ybar = (0.2126 * int(q[0]) + 0.7152 * int(q[1]) + 0.0722 * int(q[2])) * 2.0 ** -32 / n
    assert ybar < FLOOR
    e = err_gpu_formula(hs, q, n)
    assert np.isfinite(e) and e == pytest.approx(err_numpy(q, n), rel=1e-12)
    y = np.zeros(n); y[17] = 0.02
    sigma = np.sqrt(y.var(ddof=1) / n)
    assert e == pytest.approx(sigma / (2 * np.sqrt(FLOOR)), rel=1e-4)   # the floor, not the (vanishing) mean, sets the slope
    assert err_gpu_formula(hs, quantise(hs, np.zeros((n, 3), np.float32)), n) == 0.0


def test_near_cancellation_never_negative(hs):
    # a bright pixel with a spread of 1e-6: E[Y^2] - Ybar^2 cancels to the last bits of f64 (and FP32 Y rounds either way)
    rng = np.random.default_rng(3)
    for base in (1.0, 100.0, 1000.0):
        rgb = (base + rng.uniform(-1e-6, 1e-6, (500, 1)) * base).repeat(3, axis=1).astype(np.float32)
        q = quantise(hs, rgb)
        e = err_gpu_formula(hs, q, 500)
        assert e >= 0.0 and np.isfinite(e)
        assert e == pytest.approx(err_numpy(q, 500), abs=1e-12)
        ybar = base * 1.0
        assert e <= ybar * np.sqrt(2.0 ** -22 / 499) / (2 * np.sqrt(ybar))   # rounding noise of FP32 Y, as for constant samples
        assert e < 0.1 / 255


def test_ctypes_mirror_matches_header():
    hdr = open(os.path.join(ROOT, "include", "rayz_cuda.h")).read()
    assert "rayz_cuda_noise" in abi.SYMBOLS and "rayz_cuda_render_to_noise" in abi.SYMBOLS
    flags = {m.group(1): int(m.group(2)) for m in re.finditer(r"#define RZ_RENDER_([A-Z_]+)\s+(\d+)u", hdr)}
    assert flags == {"SERIAL_PASSES": abi.RENDER_SERIAL_PASSES, "MOMENTS": abi.RENDER_MOMENTS, "ACCUMULATE": abi.RENDER_ACCUMULATE}
    assert (abi.RENDER_MOMENTS, abi.RENDER_ACCUMULATE) == (2, 4)
    assert C.sizeof(abi.RzNoise) == 40
    assert [n for n, _ in abi.RzNoise._fields_] == ["samples", "n_pixels", "n_above", "mean_err", "rms_err", "max_err"]
    body = re.search(r"typedef struct RzNoise \{(.*?)\} RzNoise;", hdr, re.S).group(1)
    assert re.findall(r"\b(\w+);", body) == [n for n, _ in abi.RzNoise._fields_]
    assert abi.RzNoise.rms_err.offset == 24
    lib = abi.load()
    assert lib.rayz_cuda_abi_version() == 3


def test_params_flags():
    from rayz_b200 import Backend
    assert Backend.params(8, 8, 1).flags == 0
    assert Backend.params(8, 8, 1, moments=True).flags == 2
    assert Backend.params(8, 8, 1, accumulate=True, moments=True).flags == 6
    assert Backend.params(8, 8, 1, accumulate=True, serial_passes=True).flags == 5


def test_new_calls_fail_loudly_without_a_context():
    lib = abi.load()
    nz = abi.RzNoise()
    assert lib.rayz_cuda_noise(None, 0.01, None, C.byref(nz)) == -1
    assert b"NULL" in lib.rayz_cuda_last_error()
    p = abi.RzRenderParams()
    cam = abi.RzCamera()
    assert lib.rayz_cuda_render_to_noise(None, C.byref(cam), C.byref(p), 0.01, 64, None, None, None, C.byref(nz)) == -1
    assert b"NULL" in lib.rayz_cuda_last_error()


def test_no_gpu_means_no_progressive_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    import rayz_b200
    t = rayz_b200.random_bouncing(32, seed=42)
    with pytest.raises(abi.BackendError) as e:
        t.render(noise_target=2 / 255, max_spp=64)
    assert e.value.code == -2 and "no CPU path" in str(e.value)
