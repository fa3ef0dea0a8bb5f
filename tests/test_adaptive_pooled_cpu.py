"""CPU tests of pooled adaptive stopping (RZ_RENDER_ADAPTIVE_POOLED), compiled as host code by tests/hostsim/pooled.cu.

1. The estimator (u, the segment prior U_S with its freezing, e* with and without the RQMC gain) equals a numpy f64
   restatement of the header's formula: n < 2 pixels, all-sky segments (U_S = 0), short last segments, mixed counts.
2. The ctypes mirror, the Zig constant and the public layers carry the flag.
3. The new calls fail loudly without a context or a device."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

from rayz_b200 import _abi as abi

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
TWO32 = 2.0 ** 32


@pytest.fixture(scope="module")
def lib():
    subprocess.run(["bash", os.path.join(HERE, "hostsim", "build_pooled.sh")], check=True)
    lib = C.CDLL(os.path.join(HERE, "_build", "libhostpool.so"))
    lib.hostpool_nu0.restype = C.c_double
    lib.hostpool_u.argtypes, lib.hostpool_u.restype = [C.c_void_p, C.c_uint32], C.c_double
    lib.hostpool_err.argtypes, lib.hostpool_err.restype = [C.c_void_p, C.c_uint32, C.c_double], C.c_double
    lib.hostpool_err_rqmc.argtypes, lib.hostpool_err_rqmc.restype = [C.c_void_p, C.c_uint32, C.c_double, C.c_double], C.c_double
    lib.hostpool_pass.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32] + [C.c_void_p] * 4
    return lib


# ------------------------------------------------------------------------------- numpy restatement (include/rayz_cuda.h)
def ref_u(q, n):
    """u = n e^2 with e the iid displayed-value error of rayz_cuda_noise; 0 while n < 2 (it then takes no part)."""
    n = np.asarray(n, dtype=np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        y = (0.2126 * q[..., 0] + 0.7152 * q[..., 1] + 0.0722 * q[..., 2]) / TWO32 / n
        s2 = np.maximum(0.0, q[..., 3] / TWO32 / n - y * y) * n / (n - 1)
        e = np.sqrt(s2 / n) / (2 * np.sqrt(np.maximum(y, 1e-4)))
        return np.where(n >= 2, n * e * e, 0.0)


def ref_pool(q, counts, rows, width):
    """U_S per segment: sum d u / sum d over the pixels with n >= 2 (0 when there are none)."""
    nseg = -(-width // 64)
    lp = np.arange(rows * width)
    seg = (lp // width) * nseg + (lp % width) // 64
    d = np.where(counts >= 2, counts - 1.0, 0.0)
    du = d * ref_u(q, counts)
    num = np.bincount(seg, du, rows * nseg)
    den = np.bincount(seg, d, rows * nseg)
    return np.where(den > 0, num / np.where(den > 0, den, 1), 0.0), seg


def ref_err(q, n, pool_u, nu0, gain=None):
    n = np.asarray(n, dtype=np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        e = np.sqrt((nu0 * pool_u + (n - 1) * ref_u(q, n)) / (nu0 + n - 1) / n)
    if gain is not None:
        e = e * np.sqrt(gain)
    return np.where(n >= 2, e, np.inf)


def random_frame(rng, rows, width, counts, sky=()):
    """Sums of `counts` random paths per pixel, accum [n][4] (rgb, Y^2) in 2^-32 fixed point; the pixels in `sky` see one
    constant colour (no variance)."""
    npx = rows * width
    acc = np.zeros((npx, 4), dtype=np.uint64)
    q = lambda v: np.round(np.asarray(v, dtype=np.float64) * TWO32).astype(np.uint64)
    for lp in range(npx):
        n = int(counts[lp])
        if n == 0:
            continue
        if lp in sky:
            rgb = np.tile(np.array([0.5, 0.7, 1.0], dtype=np.float32), (n, 1))
        else:
            rgb = (rng.random((n, 3)) ** 2 * rng.choice([0.05, 1.0, 4.0])).astype(np.float32)
        y = 0.2126 * rgb[:, 0] + 0.7152 * rgb[:, 1] + 0.0722 * rgb[:, 2]
        acc[lp, :3] = q(rgb).sum(axis=0)
        acc[lp, 3] = q(y.astype(np.float64) ** 2).sum()
    return acc


def run_pass(lib, acc, counts, n, rows, width, gain=None, px_pool=None):
    nseg = -(-width // 64)
    npx = rows * width
    pool = np.full(rows * nseg, -1.0)
    px = np.full(npx, -1.0) if px_pool is None else px_pool.copy()
    err = np.zeros(npx)
    n_px = None if counts is None else np.ascontiguousarray(counts, dtype=np.uint32)
    g = None if gain is None else np.ascontiguousarray(gain, dtype=np.float64)
    lib.hostpool_pass(acc.ctypes.data, None if n_px is None else n_px.ctypes.data, n, npx, width,
                      None if g is None else g.ctypes.data, pool.ctypes.data, px.ctypes.data, err.ctypes.data)
    return pool, px, err


# ------------------------------------------------------------------------------- 1. the estimator against numpy f64
def test_nu0_is_the_documented_constant(lib):
    hdr = open(os.path.join(ROOT, "include", "rayz_cuda.h")).read()
    m = re.search(r"NU0 = (\d+)", hdr)
    assert m and float(m.group(1)) == lib.hostpool_nu0()
    dev = open(os.path.join(ROOT, "rayz_b200", "csrc", "rz_device.cuh")).read()
    assert re.search(r"#define RZ_POOL_NU0 (\d+)\.0", dev).group(1) == m.group(1)


@pytest.mark.parametrize("width", [64, 150, 200, 17])
@pytest.mark.parametrize("with_gain", [False, True])
def test_segment_prior_and_error_equal_numpy(lib, width, with_gain):
    rng = np.random.default_rng(width + 1000 * with_gain)
    rows = 3
    npx = rows * width
    counts = rng.choice([0, 1, 2, 3, 4, 8, 16, 64], npx).astype(np.uint32)   # n < 2 pixels among the others
    counts[:min(width, 64)] = rng.choice([0, 1], min(width, 64))           # a segment with no estimate at all: U_S = 0
    sky = set(range(width, width + min(width, 64)))                           # row 1's first segment: all sky
    counts[list(sky)] = rng.choice([2, 4, 8], len(sky))
    acc = random_frame(rng, rows, width, counts, sky)
    top = int(counts.max())
    gain = rng.uniform(0.2, 1.5, npx) if with_gain else None
    pool, px, err = run_pass(lib, acc, counts, top, rows, width, gain)
    want, seg = ref_pool(acc.astype(np.float64), counts.astype(np.float64), rows, width)
    np.testing.assert_allclose(pool, want, rtol=1e-12, atol=0)
    nseg = -(-width // 64)
    assert pool[0] == 0.0 and pool[nseg] == 0.0            # no pixel with two samples; all sky
    # frozen copies: the segment's U_S for the pixels at the frame's largest count, the others untouched
    at_top = counts == top
    assert np.array_equal(px[at_top], pool[seg[at_top]]) and (px[~at_top] == -1.0).all()
    # e*: over the per-pixel (frozen) priors, +inf while n < 2; the untouched -1.0 priors make the pixels below the top
    # follow the same formula with that prior, which checks that the error reads the pixel's own copy
    nu0 = lib.hostpool_nu0()
    px_ok = np.where(at_top, px, 0.25)
    _, _, err = run_pass(lib, acc, counts, top, rows, width, gain, px_pool=px_ok)
    ref = ref_err(acc.astype(np.float64), counts.astype(np.float64), px_ok, nu0, gain)
    assert np.array_equal(np.isinf(err), counts < 2) and np.array_equal(np.isinf(ref), counts < 2)
    fin = counts >= 2
    np.testing.assert_allclose(err[fin], ref[fin], rtol=1e-12)
    # the scalar forms
    for p in np.flatnonzero(fin)[::13]:
        q = np.ascontiguousarray(acc[p])
        assert lib.hostpool_u(q.ctypes.data, int(counts[p])) == pytest.approx(ref_u(acc[p].astype(np.float64), counts[p]), rel=1e-12, abs=1e-300)
        e = lib.hostpool_err(q.ctypes.data, int(counts[p]), px_ok[p])
        assert e == pytest.approx(ref_err(acc[p].astype(np.float64), counts[p], px_ok[p], nu0), rel=1e-12)
        if with_gain:
            assert lib.hostpool_err_rqmc(q.ctypes.data, int(counts[p]), px_ok[p], gain[p]) == pytest.approx(e * np.sqrt(gain[p]), rel=1e-12)


def test_uniform_frame_sky_segment_and_limits(lib):
    rng = np.random.default_rng(11)
    width, rows, n = 130, 2, 8
    sky = set(range(64))
    acc = random_frame(rng, rows, width, np.full(rows * width, n), sky)
    pool, px, err = run_pass(lib, acc, None, n, rows, width)
    want, seg = ref_pool(acc.astype(np.float64), np.full(rows * width, float(n)), rows, width)
    np.testing.assert_allclose(pool, want, rtol=1e-12)
    assert np.array_equal(px, pool[seg])                   # a uniform frame: every pixel takes its segment's prior
    assert pool[0] == 0.0 and (err[:64] == 0.0).all()      # all sky: U_S = 0 and e* = 0
    # per-pixel counts of one value equal the uniform count
    _, px2, err2 = run_pass(lib, acc, np.full(rows * width, n, dtype=np.uint32), n, rows, width)
    assert np.array_equal(px, px2) and np.array_equal(err, err2)
    # fewer than two samples: no estimate (+inf), with and without a gain
    q = np.ascontiguousarray(acc[70])
    for c in (0, 1):
        assert lib.hostpool_err(q.ctypes.data, c, 1.0) == np.inf
        assert lib.hostpool_err_rqmc(q.ctypes.data, c, 1.0, 0.0) == np.inf
    # the prior's weight: NU0 -> e* between the pixel's own error and the segment's, d = NU0 halfway in u
    u = lib.hostpool_u(q.ctypes.data, n)
    own = np.sqrt(u / n)
    for pu in (0.0, u / 4, u * 4):
        e = lib.hostpool_err(q.ctypes.data, n, pu)
        lo, hi = sorted((own, np.sqrt(pu / n)))
        assert lo - 1e-15 <= e <= hi + 1e-15


# ------------------------------------------------------------------------------- 2. the flag in every layer
def test_ctypes_mirror_and_public_layers_carry_the_flag():
    import rayz_b200
    from rayz_b200 import Backend
    hdr = open(os.path.join(ROOT, "include", "rayz_cuda.h")).read()
    m = re.search(r"#define RZ_RENDER_ADAPTIVE_POOLED\s+(0x[0-9a-fA-F]+)u", hdr)
    assert m and int(m.group(1), 0) == abi.RENDER_ADAPTIVE_POOLED == 0x40
    others = abi.RENDER_SERIAL_PASSES | abi.RENDER_MOMENTS | abi.RENDER_ACCUMULATE | abi.RENDER_ADAPTIVE | abi.RENDER_SOBOL | abi.RENDER_RQMC
    assert abi.RENDER_ADAPTIVE_POOLED & others == 0        # a bit of its own
    assert abi.load().rayz_cuda_abi_version() == 3          # additive: the ABI version stays
    zig = open(os.path.join(ROOT, "zig", "cuda_backend.zig")).read()
    assert "pub const RZ_RENDER_ADAPTIVE_POOLED: u32 = 0x40;" in zig
    host = open(os.path.join(ROOT, "host", "rayz_host.hpp")).read() + open(os.path.join(ROOT, "host", "rayz_host.cpp")).read()
    assert "RZ_RENDER_ADAPTIVE_POOLED" in host and '"--pooled"' in host
    import inspect
    assert "pooled" in inspect.signature(Backend.render_to_noise).parameters
    assert "pooled" in inspect.signature(rayz_b200.Tracer.render).parameters


# ------------------------------------------------------------------------------- 3. loud failures
def test_new_calls_fail_loudly_without_a_context():
    lib = abi.load()
    p = abi.RzRenderParams()
    p.width, p.height, p.spp, p.flags = 8, 8, 4, abi.RENDER_ADAPTIVE | abi.RENDER_ADAPTIVE_POOLED
    cam, nz = abi.RzCamera(), abi.RzNoise()
    assert lib.rayz_cuda_render_to_noise(None, C.byref(cam), C.byref(p), 0.01, 64, None, None, None, C.byref(nz)) == -1
    assert b"NULL" in lib.rayz_cuda_last_error()
    assert lib.rayz_cuda_reserve(None, C.byref(p)) == -1
    assert lib.rayz_cuda_render(None, C.byref(cam), C.byref(p), None, None, None) == -1


def test_no_gpu_means_no_pooled_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    import rayz_b200
    t = rayz_b200.random_bouncing(32, seed=42)
    with pytest.raises(abi.BackendError) as e:
        t.render(noise_target=2 / 255, max_spp=64, adaptive=True, pooled=True)
    assert e.value.code == -2 and "no CPU path" in str(e.value)
    assert t.pixel_samples is None and t.noise is None
