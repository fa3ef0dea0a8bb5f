"""CPU tests of the denoiser (rayz_cuda_denoise): the ctypes mirror of RzDenoiseParams and the prototype against
include/rayz_cuda.h and the Zig externs, loud failures without a context or a device, the per-tap weight and the
(de)modulation of rz_denoise.cuh compiled as host code (tests/hostsim/denoise.cu) against a numpy f64 restatement, and the
properties of the numpy reference filter that tests/test_denoise_gpu.py compares the GPU with.

The reference below is the contract of include/rayz_cuda.h (rayz_cuda_denoise) in f64, on the public readouts: the resolved
linear frame, rayz_cuda_noise's error and the guide buffers."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

from rayz_b200 import _abi as abi

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)

LUMA = np.array([0.2126, 0.7152, 0.0722])
H5 = np.array([1.0, 4.0, 6.0, 4.0, 1.0]) / 16.0
ALBEDO_FLOOR, LUM_EPS, DEPTH_EPS, Y_FLOOR = 1e-3, 1e-4, 1e-2, 1e-4


def weight_ref(yp, yq, gv, n_p, n_q, gp, ox, oy, sl, sn, sz):
    """w_l w_n w_z of include/rayz_cuda.h in f64 (arrays broadcast; n_*: [..., 4] normal xyz + depth, gp: [..., 2])."""
    with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
        wl = np.exp(-np.abs(yp - yq) / (sl * np.sqrt(gv) + LUM_EPS))
        pp = (n_p[..., :3] ** 2).sum(-1)
        qq = (n_q[..., :3] ** 2).sum(-1)
        both = (pp > 0) & (qq > 0)
        c = (n_p[..., :3] * n_q[..., :3]).sum(-1) / np.sqrt(np.where(both, pp * qq, 1.0))
        wn = np.where(both, np.clip(c, 0.0, 1.0) ** sn, np.where((pp > 0) == (qq > 0), 1.0, 0.0))
        wz = np.exp(-np.abs(n_p[..., 3] - n_q[..., 3]) / (sz * np.abs(gp[..., 0] * ox + gp[..., 1] * oy) + DEPTH_EPS))
    return wl * wn * wz


def demodulate_ref(c, e, a):
    """(i, v) of include/rayz_cuda.h in f64: c [..., 3] linear rgb, e [...] error, a [..., 3] albedo."""
    with np.errstate(invalid="ignore", over="ignore"):
        v = 4.0 * e * e * np.maximum(c @ LUMA, Y_FLOOR)
        return c / np.maximum(a, ALBEDO_FLOOR), v / np.maximum(a @ LUMA, ALBEDO_FLOOR) ** 2


def _shift(x, dy, dx):
    """x[y + dy, x + dx] for every pixel (indices clamped) and whether that tap is inside the frame."""
    h, w = x.shape[:2]
    ys, xs = np.arange(h) + dy, np.arange(w) + dx
    inside = ((ys >= 0) & (ys < h))[:, None] & ((xs >= 0) & (xs < w))[None, :]
    return x[np.clip(ys, 0, h - 1)][:, np.clip(xs, 0, w - 1)], inside


def denoise_ref(lin, err, albedo, normal, iterations=5, sigma_luminance=4.0, sigma_normal=128.0, sigma_depth=1.0,
                return_variance=False):
    """The filter of include/rayz_cuda.h (rayz_cuda_denoise) in numpy f64 on an [h, w] frame: lin [h,w,4] (or 3), err [h,w],
    albedo [h,w,4] (rgb used), normal [h,w,4] (xyz normal, w depth) -> denoised linear rgb [h,w,3] f64 (and, with
    return_variance and iterations > 0, the last level's demodulated variance v' [h,w])."""
    c = np.asarray(lin, dtype=np.float64)[..., :3]
    if iterations == 0:
        return c
    a = np.asarray(albedo, dtype=np.float64)[..., :3]
    nrm = np.asarray(normal, dtype=np.float64)
    i, v = demodulate_ref(c, np.asarray(err, dtype=np.float64), a)
    z = nrm[..., 3]
    h, w = z.shape
    xs, ys = np.arange(w), np.arange(h)
    gx = (z[:, np.minimum(xs + 1, w - 1)] - z[:, np.maximum(xs - 1, 0)]) / 2
    gy = (z[np.minimum(ys + 1, h - 1)] - z[np.maximum(ys - 1, 0)]) / 2
    g = np.stack([gx, gy], axis=-1)
    for k in range(iterations):
        s = 1 << k
        num = np.zeros((h, w))
        den = np.zeros((h, w))
        for dy in (-1, 0, 1):
            for dx in (-1, 0, 1):
                vq, inside = _shift(v, dy, dx)
                kk = (2 - dx * dx) * (2 - dy * dy)
                num += np.where(inside, kk * vq, 0.0)
                den += np.where(inside, kk, 0.0)
        gv = num / den
        yi = i @ LUMA
        sw, si, sv = np.zeros((h, w)), np.zeros((h, w, 3)), np.zeros((h, w))
        for dy in range(-2, 3):
            for dx in range(-2, 3):
                iq, inside = _shift(i, dy * s, dx * s)
                vq, _ = _shift(v, dy * s, dx * s)
                nq, _ = _shift(nrm, dy * s, dx * s)
                wt = H5[dx + 2] * H5[dy + 2] * weight_ref(yi, iq @ LUMA, gv, nrm, nq, g, dx * s, dy * s,
                                                          sigma_luminance, sigma_normal, sigma_depth)
                wt = np.where(inside, wt, 0.0)
                sw += wt
                si += wt[..., None] * iq
                w2 = wt * wt
                w32 = wt.astype(np.float32)
                with np.errstate(invalid="ignore", under="ignore"):
                    sv += np.where(w32 * w32 > 0, w2 * vq, 0.0)   # the contract's guard: the f32 w^2
        i, v = si / sw[..., None], sv / (sw * sw)
    out = i * np.maximum(a, ALBEDO_FLOOR)
    return (out, v) if return_variance else out


def quantise_ref(x):
    """writePPM's transform in f64 of f32 linear values: trunc(255 clamp(sqrt(x), 0, 1)) (sqrt of x <= 0 is 0)."""
    x = np.asarray(x, dtype=np.float64)
    return np.trunc(np.clip(np.sqrt(np.maximum(x, 0.0)), 0.0, 1.0) * 255.0).astype(np.uint8)


# ------------------------------------------------------------------------------- ABI
def test_ctypes_struct_and_prototype_match_header():
    hdr = open(os.path.join(ROOT, "include", "rayz_cuda.h")).read()
    body = re.search(r"typedef struct RzDenoiseParams \{(.*?)\} RzDenoiseParams;", hdr, re.S).group(1)
    fields = re.findall(r"^\s*(uint32_t|float)\s+(\w+);", body, re.M)
    ctype = {"uint32_t": C.c_uint32, "float": C.c_float}
    assert [(n, ctype[t]) for t, n in fields] == list(abi.RzDenoiseParams._fields_)
    assert C.sizeof(abi.RzDenoiseParams) == 24
    assert [getattr(abi.RzDenoiseParams, n).offset for n, _ in abi.RzDenoiseParams._fields_] == [0, 4, 8, 12, 16, 20]
    proto = re.search(r"int rayz_cuda_denoise\(([^)]*)\);", hdr)
    assert proto and [a.strip() for a in proto.group(1).split(",")] == [
        "RzContext *ctx", "const RzDenoiseParams *dp", "float *out_linear_rgba", "uint8_t *out_rgb8"]
    res, args = abi.SYMBOLS["rayz_cuda_denoise"]
    assert res is C.c_int and args == [C.c_void_p, C.POINTER(abi.RzDenoiseParams), C.c_void_p, C.c_void_p]
    assert re.search(r"#define RAYZ_CUDA_ABI_VERSION 3\b", hdr)
    assert abi.load().rayz_cuda_abi_version() == 3
    zig = open(os.path.join(ROOT, "zig", "cuda_backend.zig")).read()
    assert "pub extern fn rayz_cuda_denoise(ctx: *RzContext, dp: ?*const RzDenoiseParams, out_linear_rgba: ?[*]f32, " \
           "out_rgb8: ?[*]u8) c_int;" in zig
    zs = re.search(r"pub const RzDenoiseParams = extern struct \{(.*?)\n\};", zig, re.S).group(1)
    assert re.findall(r"^\s*(\w+): (u32|f32)", zs, re.M) == [(n, {"uint32_t": "u32", "float": "f32"}[t]) for t, n in fields]


def test_denoise_fails_loudly_without_a_context():
    lib = abi.load()
    out = np.zeros(8 * 4, dtype=np.float32)
    assert lib.rayz_cuda_denoise(None, None, out.ctypes.data, None) == -1
    assert lib.rayz_cuda_last_error().startswith(b"denoise:") and b"NULL" in lib.rayz_cuda_last_error()
    assert (out == 0).all()


def test_no_gpu_means_no_denoise_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    import rayz_b200
    t = rayz_b200.random_bouncing(32, seed=42)
    with pytest.raises(abi.BackendError) as e:
        t.denoise()
    assert e.value.code == -2 and "no CPU path" in str(e.value)
    assert t.denoised is None


# ------------------------------------------------------------------------------- rz_denoise.cuh as host code
@pytest.fixture(scope="module")
def hd():
    subprocess.run(["bash", os.path.join(HERE, "hostsim", "build_denoise.sh")], check=True)
    lib = C.CDLL(os.path.join(HERE, "_build", "libhostdenoise.so"))
    lib.hostdenoise_weights.argtypes = [C.c_void_p] * 3 + [C.c_uint32, C.c_void_p]
    lib.hostdenoise_demodulate.argtypes = [C.c_void_p] * 3 + [C.c_uint32, C.c_void_p, C.c_void_p]
    return lib


def _unit_ish(rng, n):
    d = rng.normal(size=(n, 3))
    return d / np.linalg.norm(d, axis=1, keepdims=True) * rng.uniform(0.3, 1.0, size=(n, 1))


def test_weight_matches_f64_restatement(hd):
    rng = np.random.default_rng(7)
    n = 20000
    t = np.zeros((n, 11), dtype=np.float32)
    t[:, 0], t[:, 1] = rng.uniform(0, 2, n), rng.uniform(0, 2, n)
    t[:, 2] = rng.uniform(0, 0.05, n) ** 2
    t[:, 3:6], t[:, 7:10] = _unit_ish(rng, n), _unit_ish(rng, n)
    t[:, 6], t[:, 10] = rng.uniform(0, 20, n), rng.uniform(0, 20, n)
    near = rng.random(n) < 0.5   # half of the taps on the same surface: similar normal and depth, weights far from 0
    t[near, 7:10] = t[near, 3:6] + rng.normal(scale=0.02, size=(near.sum(), 3))
    t[near, 10] = t[near, 6] + rng.normal(scale=0.05, size=near.sum())
    t[near, 1] = t[near, 0] + rng.normal(scale=0.01, size=near.sum())
    # edge cases: v = +inf, zero normals on one or both sides, z = 0
    t[:50, 2] = np.inf
    t[50:100, 3:6] = 0
    t[100:150, 7:10] = 0
    t[150:200, 3:6] = 0
    t[150:200, 7:10] = 0
    t[200:250, 6] = 0
    t[250:300, 10] = 0
    o = np.zeros((n, 4), dtype=np.float32)
    o[:, :2] = rng.uniform(-1, 1, size=(n, 2))
    step = 2 ** rng.integers(0, 5, n)
    o[:, 2], o[:, 3] = rng.integers(-2, 3, n) * step, rng.integers(-2, 3, n) * step
    for sig in ((4.0, 128.0, 1.0), (1.0, 32.0, 0.25), (10.0, 1.0, 4.0)):
        s = np.array(sig, dtype=np.float32)
        got = np.empty(n, dtype=np.float32)
        hd.hostdenoise_weights(t.ctypes.data, o.ctypes.data, s.ctypes.data, n, got.ctypes.data)
        t64, o64 = t.astype(np.float64), o.astype(np.float64)
        want = weight_ref(t64[:, 0], t64[:, 1], t64[:, 2], t64[:, 3:7], t64[:, 7:11], o64[:, :2], o64[:, 2], o64[:, 3], *sig)
        # f32 exp and pow of arguments rounded to f32: a relative error of a few ulp times the size of the exponent, plus the
        # cosine's absolute rounding error (a few ulp of |n_p| |n_q|, however small the cosine is) raised to the power sigma_n
        expo = -np.log(np.maximum(want, 1e-300))
        n_p, n_q = t64[:, 3:6], t64[:, 7:10]
        with np.errstate(invalid="ignore", divide="ignore"):
            cos = (n_p * n_q).sum(1) / np.sqrt((n_p ** 2).sum(1) * (n_q ** 2).sum(1))
            cos_term = np.where(cos > 0, sig[1] / np.where(cos > 0, cos, 1.0), 0.0)
        assert (np.abs(got - want) <= 4e-7 * (8 + expo + cos_term) * want + 1e-37).all(), sig
        e = t64[:50]   # w_l = 1 at v = inf: the weight of the same tap with equal luminances
        assert (want[:50] == weight_ref(e[:, 1], e[:, 1], e[:, 2], e[:, 3:7], e[:, 7:11], o64[:50, :2],
                                                                  o64[:50, 2], o64[:50, 3], *sig)).all()
        assert (got[50:150] == 0).all() and (want[50:150] == 0).all()   # a zero normal on one side only
        b = t64[150:200]   # both zero (sky and sky): w_n = 1, the weight is w_l w_z
        wl = np.exp(-np.abs(b[:, 0] - b[:, 1]) / (sig[0] * np.sqrt(b[:, 2]) + 1e-4))
        wz = np.exp(-np.abs(b[:, 6] - b[:, 10]) / (sig[2] * np.abs(o64[150:200, 0] * o64[150:200, 2] + o64[150:200, 1] * o64[150:200, 3]) + 1e-2))
        assert (want[150:200] == wl * wz).all()
        assert ((want > 0.1) & (want < 0.9)).sum() > 1000


def test_demodulate_and_remodulate_match_f64(hd):
    rng = np.random.default_rng(11)
    n = 5000
    c = np.concatenate([rng.uniform(0, 3, (n, 3)), np.ones((n, 1))], axis=1).astype(np.float32)
    e = rng.uniform(0, 0.05, n).astype(np.float32)
    e[:20] = np.inf
    a = np.concatenate([rng.uniform(0, 1, (n, 3)), rng.uniform(0, 1, (n, 1))], axis=1).astype(np.float32)
    a[20:60, :3] = rng.uniform(0, 1e-3, (40, 3))          # albedo below the floor
    a[60:80, :3] = 0
    iv = np.empty((n, 4), dtype=np.float32)
    rm = np.empty((n, 4), dtype=np.float32)
    hd.hostdenoise_demodulate(c.ctypes.data, e.ctypes.data, a.ctypes.data, n, iv.ctypes.data, rm.ctypes.data)
    i, v = demodulate_ref(c[:, :3].astype(np.float64), e.astype(np.float64), a[:, :3].astype(np.float64))
    assert np.allclose(iv[:, :3], i, rtol=3e-7, atol=0)
    assert np.isinf(iv[:20, 3]).all() and np.isinf(v[:20]).all()
    assert np.allclose(iv[20:, 3], v[20:], rtol=2e-6, atol=0)
    assert np.allclose(rm[:, :3], i * np.maximum(a[:, :3], 1e-3), rtol=5e-7, atol=0) and (rm[:, 3] == 1).all()
    assert np.allclose(rm[:, :3], c[:, :3], rtol=5e-7, atol=0)   # remodulation undoes demodulation


# ------------------------------------------------------------------------------- the numpy reference filter
def _frame(rng, h=23, w=31):
    lin = rng.uniform(0, 1, (h, w, 4))
    err = rng.uniform(0, 0.05, (h, w))
    alb = rng.uniform(0, 1, (h, w, 4))
    nrm = np.concatenate([_unit_ish(rng, h * w).reshape(h, w, 3), rng.uniform(1, 5, (h, w, 1))], axis=-1)
    nrm[:3, :5, :] = 0   # a patch of sky
    return lin, err, alb, nrm


def test_reference_keeps_a_constant_image():
    h, w = 17, 29
    lin = np.broadcast_to(np.array([0.3, 0.5, 0.2, 1.0]), (h, w, 4))
    alb = np.broadcast_to(np.array([0.6, 0.4, 0.5, 1.0]), (h, w, 4))
    nrm = np.broadcast_to(np.array([0.0, 0.6, 0.8, 3.0]), (h, w, 4))
    out = denoise_ref(lin, np.full((h, w), 0.02), alb, nrm, iterations=5)
    assert np.allclose(out, lin[..., :3], rtol=1e-13, atol=0)


@pytest.mark.parametrize("iterations", [1, 3, 5])
def test_reference_is_symmetric_under_mirroring(iterations):
    lin, err, alb, nrm = _frame(np.random.default_rng(iterations))
    out = denoise_ref(lin, err, alb, nrm, iterations)
    assert np.allclose(denoise_ref(lin[:, ::-1], err[:, ::-1], alb[:, ::-1], nrm[:, ::-1], iterations)[:, ::-1], out, rtol=1e-12, atol=1e-15)
    assert np.allclose(denoise_ref(lin[::-1], err[::-1], alb[::-1], nrm[::-1], iterations)[::-1], out, rtol=1e-12, atol=1e-15)
    assert not np.allclose(out, lin[..., :3])   # the filter did something


def test_reference_variance_guard_is_the_f32_square():
    """A tap with v = +inf whose weight is positive but whose f32 w^2 is 0 adds nothing to the variance.  1 x 3 frame, depth
    (2, 1, 2): the centre's depth gradient is 0, so each side tap has w_z = exp(-1 / 1e-2) and w = 0.094 e^-100 = 3.5e-45,
    whose square is 1.2e-89 in f64 but 0 in f32.  The side pixels have n < 2 (e = +inf); the centre keeps a finite v'."""
    lin = np.full((1, 3, 4), 0.5)
    alb = np.full((1, 3, 4), 0.5)
    err = np.array([[np.inf, 0.01, np.inf]])
    nrm = np.zeros((1, 3, 4))
    nrm[..., 2] = 1.0
    nrm[0, :, 3] = (2.0, 1.0, 2.0)
    w_side = H5[1] * H5[2] * np.exp(-1.0 / DEPTH_EPS)
    assert w_side * w_side > 0 and np.float32(w_side) > 0 and np.float32(w_side) * np.float32(w_side) == 0
    _, v = denoise_ref(lin, err, alb, nrm, iterations=1, return_variance=True)
    assert np.isinf(v[0, 0]) and np.isinf(v[0, 2])
    assert np.isfinite(v[0, 1]) and v[0, 1] > 0


def test_reference_at_zero_iterations_is_the_input():
    lin, err, alb, nrm = _frame(np.random.default_rng(3))
    assert np.array_equal(denoise_ref(lin, err, alb, nrm, 0), lin[..., :3])


def test_quantise_ref_matches_the_resolve_transform():
    x = np.array([-1.0, 0.0, 1e-9, 0.25, 1.0, 4.0, (254.5 / 255) ** 2], dtype=np.float32)
    assert quantise_ref(x).tolist() == [0, 0, 0, 127, 255, 255, 254]
