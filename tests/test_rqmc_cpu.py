"""CPU tests of the randomised-QMC noise estimate (RZ_RENDER_RQMC), compiled as host code by tests/hostsim/rqmc.cu.

1. The replicate mapping of rz_sobol_pair equals a numpy restatement (test_sampler_cpu.py's, plus the replicate seed step),
   and with the flag off it is today's rz_sobol_pair.
2. Each replicate's aligned blocks are (0,k,2)-nets; the two replicates are decorrelated.
3. The replicate terms, the segment gain and rz_pixel_err_rqmc equal numpy f64.
4. Backend.params and Tracer.sampler build the flag bits without a device."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
from scipy import stats

from test_sampler_cpu import hash32, owen, sobol

HERE = os.path.dirname(os.path.abspath(__file__))
TWO32 = 2.0 ** 32


@pytest.fixture(scope="module")
def lib():
    subprocess.run(["bash", os.path.join(HERE, "hostsim", "build_rqmc.sh")], check=True)
    lib = C.CDLL(os.path.join(HERE, "_build", "libhostrqmc.so"))
    lib.hostrqmc_pairs.argtypes = [C.c_uint64, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]
    lib.hostrqmc_rep_sums.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p]
    for f in (lib.hostrqmc_var_iid, lib.hostrqmc_var_rep):
        f.argtypes, f.restype = [C.c_void_p, C.c_uint32], C.c_double
    lib.hostrqmc_err.argtypes, lib.hostrqmc_err.restype = [C.c_void_p, C.c_uint32, C.c_double], C.c_double
    lib.hostrqmc_segments.argtypes, lib.hostrqmc_segments.restype = [C.c_uint32], C.c_uint32
    lib.hostrqmc_segment_of.argtypes, lib.hostrqmc_segment_of.restype = [C.c_uint32, C.c_uint32], C.c_uint64
    lib.hostrqmc_gains.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p]
    return lib


def pairs(lib, seed, gpix, pair, sample, rqmc=True):
    g, p, s = (np.ascontiguousarray(x, dtype=np.uint32) for x in np.broadcast_arrays(gpix, pair, sample))
    xy = np.zeros((g.size, 2), dtype=np.uint32)
    lib.hostrqmc_pairs(seed, int(rqmc), g.ctypes.data, p.ctypes.data, s.ctypes.data, g.size, xy.ctypes.data)
    return xy


def ref_pairs(seed, gpix, pair, sample, rqmc=True):
    """test_sampler_cpu.ref_pairs with the header's replicate step: b_r = hash32(b ^ (0x9e3779b9 + r)), index i >> 1."""
    g, p, s = (np.asarray(x, dtype=np.uint64) for x in np.broadcast_arrays(gpix, pair, sample))
    k0, k1 = np.uint64(seed & 0xFFFFFFFF), np.uint64(seed >> 32)
    h = hash32(np.full(g.shape, k0 ^ np.uint64(0x6a09e667), dtype=np.uint64))
    h = hash32(h ^ k1)
    h = hash32(h ^ g)
    base = hash32(h ^ p)
    if rqmc:
        base = hash32(base ^ (np.uint64(0x9e3779b9) + (s & np.uint64(1))))
        s = s >> np.uint64(1)
    i = owen(s, hash32(base))
    x = owen(sobol(i, 0), hash32(base ^ np.uint64(1)))
    y = owen(sobol(i, 1), hash32(base ^ np.uint64(2)))
    return np.stack([x, y], axis=-1).astype(np.uint32)


# ------------------------------------------------------------------------------- 1. the replicate mapping, bit-exact
@pytest.mark.parametrize("seed", [0, 7, 0xDEADBEEFCAFEF00D])
def test_replicate_mapping_equals_numpy_restatement(lib, seed):
    rng = np.random.default_rng(seed & 0xFFFF)
    n = 3000
    gpix = np.concatenate([rng.integers(0, 1 << 32, n // 2, dtype=np.uint64), np.array([0, 1, (1 << 32) - 1] * (n // 2), dtype=np.uint64)])[:n]
    pair = rng.integers(0, 60, n, dtype=np.uint64)
    sample = np.concatenate([rng.integers(0, 1 << 32, n // 2, dtype=np.uint64), np.arange(n // 4, dtype=np.uint64),
                             np.array([(1 << 32) - 1, (1 << 32) - 2, 0, 1, 2, 3] * (n // 20), dtype=np.uint64)])[:n]
    assert np.array_equal(pairs(lib, seed, gpix, pair, sample), ref_pairs(seed, gpix, pair, sample))
    # without the flag: today's rz_sobol_pair, bit for bit
    assert np.array_equal(pairs(lib, seed, gpix, pair, sample, rqmc=False), ref_pairs(seed, gpix, pair, sample, rqmc=False))


# ------------------------------------------------------------------------------- 2. stratification and decorrelation
@pytest.mark.parametrize("gpix,pair", [(0, 0), (123457, 1), (0xFFFFFFFF, 9), (2024, 52)])
@pytest.mark.parametrize("r", [0, 1])
def test_each_replicate_s_aligned_blocks_are_0k2_nets(lib, gpix, pair, r):
    """Replicate r's samples j in [m 2^k, (m + 1) 2^k), i.e. sample indices 2 j + r, form a (0,k,2)-net for k = 0..12."""
    for k in range(13):
        for m in (0, 1, 3, (1 << (19 - k)) + 5, ((1 << 31) >> k) - 1):
            j = np.arange(m << k, (m + 1) << k, dtype=np.uint64)
            q = (pairs(lib, 99, gpix, pair, 2 * j + r) >> 8).astype(np.int64)
            for a in range(k + 1):
                b = k - a
                cell = (q[:, 0] >> (24 - a)) << b | (q[:, 1] >> (24 - b))
                assert len(np.unique(cell)) == 1 << k, (k, m, a)


def test_replicates_are_decorrelated(lib):
    s = np.arange(4096)
    r0 = (pairs(lib, 5, 31337, 0, 2 * s)[:, 0] >> 8).astype(np.float64)
    r1 = (pairs(lib, 5, 31337, 0, 2 * s + 1)[:, 0] >> 8).astype(np.float64)
    assert abs(np.corrcoef(r0, r1)[0, 1]) < 0.05
    assert (r0 != r1).mean() > 0.99
    # the first samples of many pixels, in each replicate, are uniform; other pairs of the same pixel are uncorrelated
    for r in (0, 1):
        u = (pairs(lib, 5, np.arange(4096), 0, r) >> 8).astype(np.float64) / 2.0 ** 24
        for c in range(2):
            assert stats.kstest(u[:, c], "uniform").pvalue > 0.01
        x = [(pairs(lib, 5, 31337, p, 2 * s + r)[:, 0] >> 8).astype(np.float64) for p in (0, 1, 3)]
        for i in range(3):
            for j in range(i + 1, 3):
                assert abs(np.corrcoef(x[i], x[j])[0, 1]) < 0.05, (r, i, j)


# ------------------------------------------------------------------------------- 3. the estimate against numpy f64
def ref_var_iid(q, n):
    y = (0.2126 * q[..., 0] + 0.7152 * q[..., 1] + 0.0722 * q[..., 2]) / TWO32 / n
    s2 = np.maximum(0.0, q[..., 3] / TWO32 / n - y * y) * n / (n - 1)
    return s2 / n


def ref_var_rep(r, n):
    m = n / 2
    return (r[..., 0] / TWO32 / m - r[..., 1] / TWO32 / m) ** 2 / 4


def random_frame(rng, rows, width, counts):
    """Sums of `counts` random paths per pixel: accum [n][4] (rgb, Y^2) and rep [n][2] (Y per replicate), uint64."""
    npx = rows * width
    acc = np.zeros((npx, 4), dtype=np.uint64)
    rep = np.zeros((npx, 2), dtype=np.uint64)
    for lp in range(npx):
        n = int(counts[lp])
        rgb = (rng.random((n, 3)) ** 2 * rng.choice([0.2, 1.0, 3.0])).astype(np.float32)
        y = (0.2126 * rgb[:, 0] + 0.7152 * rgb[:, 1] + 0.0722 * rgb[:, 2])
        q = lambda v: np.round(v.astype(np.float64) * TWO32).astype(np.uint64)
        acc[lp, :3] = q(rgb).sum(axis=0)
        acc[lp, 3] = q(y * y).sum()
        rep[lp, 0], rep[lp, 1] = q(y[0::2]).sum(), q(y[1::2]).sum()
    return acc, rep


def test_replicate_sums_follow_the_sample_parity(lib):
    rng = np.random.default_rng(3)
    rgb = (rng.random((10, 3)) * 2).astype(np.float32)
    one = np.zeros((10, 2), dtype=np.uint64)
    for k in range(10):                                      # each path alone: its fixed-point clamped luminance, in slot 0
        lib.hostrqmc_rep_sums(np.ascontiguousarray(rgb[k]).ctypes.data, 1, 0, one[k].ctypes.data)
    y = rgb.astype(np.float64) @ np.array([0.2126, 0.7152, 0.0722])
    np.testing.assert_allclose(one[:, 0].astype(np.float64) / TWO32, y, rtol=1e-6)
    assert (one[:, 1] == 0).all()
    for off in (0, 1, 4, 7):                                 # path k of a batch starting at sample `off` is replicate (off + k) & 1
        out = np.zeros(2, dtype=np.uint64)
        lib.hostrqmc_rep_sums(rgb.ctypes.data, 10, off, out.ctypes.data)
        par = (off + np.arange(10)) & 1
        assert out[0] == one[par == 0, 0].sum() and out[1] == one[par == 1, 0].sum(), off


@pytest.mark.parametrize("width", [64, 150, 200, 17])
def test_segment_gain_and_error_equal_numpy(lib, width):
    rng = np.random.default_rng(width)
    rows = 3
    npx = rows * width
    nseg = -(-width // 64)
    assert lib.hostrqmc_segments(width) == nseg
    counts = 2 * rng.integers(1, 12, npx)                   # different (even) counts in one segment
    acc, rep = random_frame(rng, rows, width, counts)
    n_px = counts.astype(np.uint32)
    gain, px = np.zeros(rows * nseg), np.full(npx, -1.0)
    top = int(counts.max())
    lib.hostrqmc_gains(acc.ctypes.data, rep.ctypes.data, n_px.ctypes.data, top, npx, width, gain.ctypes.data, px.ctypes.data)
    af, rf, nf = acc.astype(np.float64), rep.astype(np.float64), counts.astype(np.float64)
    v_iid, v_rep = ref_var_iid(af, nf), ref_var_rep(rf, nf)
    lp = np.arange(npx)
    seg = (lp // width) * nseg + (lp % width) // 64          # the last segment of a row is the short one
    assert all(lib.hostrqmc_segment_of(int(p), width) == s for p, s in zip(lp[::7], seg[::7]))
    want = np.array([v_rep[seg == s].sum() / v_iid[seg == s].sum() for s in range(rows * nseg)])
    np.testing.assert_allclose(gain, want, rtol=1e-12)
    # the per-pixel gains: the segment's for the pixels at the frame's largest count, the others untouched (frozen)
    assert np.array_equal(px[counts == top], gain[seg[counts == top]]) and (px[counts != top] == -1.0).all()
    for p in lp[::11]:
        assert lib.hostrqmc_var_iid(acc[p].ctypes.data, int(counts[p])) == pytest.approx(v_iid[p], rel=1e-12)
        assert lib.hostrqmc_var_rep(rep[p].ctypes.data, int(counts[p])) == pytest.approx(v_rep[p], rel=1e-12, abs=1e-300)
        y = (0.2126 * af[p, 0] + 0.7152 * af[p, 1] + 0.0722 * af[p, 2]) / TWO32 / nf[p]
        e_iid = np.sqrt(v_iid[p]) / (2 * np.sqrt(max(y, 1e-4)))
        assert lib.hostrqmc_err(acc[p].ctypes.data, int(counts[p]), gain[seg[p]]) == pytest.approx(e_iid * np.sqrt(want[seg[p]]), rel=1e-12)


def test_uniform_count_and_zero_denominator(lib):
    rng = np.random.default_rng(9)
    width, rows, n = 130, 2, 8
    acc, rep = random_frame(rng, rows, width, np.full(rows * width, n))
    # the first segment of row 1: every path the same value -> V_iid = 0 and V_rep = 0 -> G = 1
    flat = slice(width, width + 64)
    acc[flat, :3] = np.uint64(n) * np.uint64(1 << 31)
    acc[flat, 3] = np.uint64(n) * np.uint64(1 << 30)        # Y = 0.5 for every path: Y^2 = 0.25
    rep[flat] = np.uint64(n // 2) * np.uint64(1 << 31)
    gain, px = np.zeros(rows * 3), np.zeros(rows * width)
    lib.hostrqmc_gains(acc.ctypes.data, rep.ctypes.data, None, n, rows * width, width, gain.ctypes.data, px.ctypes.data)
    assert np.array_equal(px, gain[(np.arange(rows * width) // width) * 3 + (np.arange(rows * width) % width) // 64])   # uniform: all
    assert gain[3] == 1.0
    g2, px2 = np.zeros_like(gain), np.zeros_like(px)
    counts = np.full(rows * width, n, dtype=np.uint32)
    lib.hostrqmc_gains(acc.ctypes.data, rep.ctypes.data, counts.ctypes.data, n, rows * width, width, g2.ctypes.data, px2.ctypes.data)
    assert np.array_equal(px, px2)
    assert np.array_equal(gain, g2)                          # a uniform count equals per-pixel counts of that value
    assert (gain[[0, 1, 2, 4, 5]] > 0).all() and np.isfinite(gain).all()
    # fewer than two samples: no estimate (+inf), as rz_pixel_err
    assert lib.hostrqmc_err(acc[0].ctypes.data, 1, 0.5) == np.inf
    assert lib.hostrqmc_err(acc[0].ctypes.data, 0, 0.0) == np.inf


# ------------------------------------------------------------------------------- 4. flag bits without a device
def test_flag_bits():
    from rayz_b200 import _abi as abi
    from rayz_b200 import Backend
    import rayz_b200
    assert abi.RENDER_RQMC == 0x20
    assert Backend.params(8, 8, 2, rqmc=True).flags == abi.RENDER_RQMC          # no implied bits: the library refuses it alone
    assert Backend.params(8, 8, 2, sobol=True, rqmc=True, moments=True).flags == abi.RENDER_SOBOL | abi.RENDER_RQMC | abi.RENDER_MOMENTS
    with open(os.path.join(HERE, "..", "include", "rayz_cuda.h")) as f:
        assert "#define RZ_RENDER_RQMC 0x20u" in f.read()
    with open(os.path.join(HERE, "..", "zig", "cuda_backend.zig")) as f:
        assert "pub const RZ_RENDER_RQMC: u32 = 0x20;" in f.read()
    t = rayz_b200.random_bouncing(32, seed=1)
    want = {"philox": {}, "sobol": {"sobol": True}, "sobol-rqmc": {"sobol": True, "rqmc": True, "moments": True}}
    for name, kw in want.items():
        t.sampler = name
        assert t._sampler() == kw
        assert Backend.params(8, 8, 2, **t._sampler()).flags == Backend.params(8, 8, 2, **kw).flags
    t.sampler = "halton"
    with pytest.raises(ValueError, match="'philox', 'sobol' or 'sobol-rqmc'"):
        t._sampler()
