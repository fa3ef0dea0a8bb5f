"""CPU tests of the low-discrepancy sampler (rz_sampler.cuh, RZ_RENDER_SOBOL), compiled as host code by tests/hostsim/sampler.cu.

1. It equals an independent numpy uint32 restatement: Sobol dimensions 0 and 1 built from the direction numbers, the
   nested-uniform scramble and the seed derivation.
2. The stratification the header promises: every aligned block of 2^k samples of a pair is a (0,k,2)-net.
3. Different pixels and different pairs are decorrelated."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
from scipy import stats

HERE = os.path.dirname(os.path.abspath(__file__))
M32 = np.uint64(0xFFFFFFFF)


@pytest.fixture(scope="module")
def lib():
    subprocess.run(["bash", os.path.join(HERE, "hostsim", "build_sampler.sh")], check=True)
    lib = C.CDLL(os.path.join(HERE, "_build", "libhostsampler.so"))
    lib.hostsampler_pairs.argtypes = [C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p]
    lib.hostsampler_uniforms.argtypes = [C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p]
    return lib


def pairs(lib, seed, gpix, pair, sample):
    """(n, 2) uint32 coordinates and (n,) base seeds of the host-compiled sampler; gpix, pair, sample broadcast together."""
    g, p, s = (np.ascontiguousarray(x, dtype=np.uint32) for x in np.broadcast_arrays(gpix, pair, sample))
    n = g.size
    xy = np.zeros((n, 2), dtype=np.uint32)
    base = np.zeros(n, dtype=np.uint32)
    lib.hostsampler_pairs(seed, g.ctypes.data, p.ctypes.data, s.ctypes.data, n, xy.ctypes.data, base.ctypes.data)
    return xy, base


# ------------------------------------------------------------------------------- numpy restatement (uint64 arithmetic, masked)
def mul32(a, b):
    return (a.astype(np.uint64) * np.uint64(b)) & M32


def hash32(x):
    x = x.astype(np.uint64)
    x ^= x >> np.uint64(16)
    x = mul32(x, 0x7feb352d)
    x ^= x >> np.uint64(15)
    x = mul32(x, 0x846ca68b)
    x ^= x >> np.uint64(16)
    return x


def brev(x):
    x = x.astype(np.uint64)
    out = np.zeros_like(x)
    for b in range(32):
        out |= ((x >> np.uint64(b)) & np.uint64(1)) << np.uint64(31 - b)
    return out


def owen(x, seed):
    """Nested-uniform scramble: bit reversal, Laine-Karras-style hash keyed by seed, bit reversal."""
    x = brev(x)
    x = (x + seed) & M32
    for c in (0x6c50b47c, 0xb82f1e52, 0xc7afe638, 0x8d22f6e6):
        x ^= mul32(x, c)
    return brev(x)


def direction_numbers():
    """Joe-Kuo d = 2 (s = 1, a = 0, m_1 = 1): m_j = 2 m_{j-1} xor m_{j-1}; V_j = m_j 2^(32 - j), j = 1..32."""
    m = [1]
    for _ in range(31):
        m.append((2 * m[-1]) ^ m[-1])
    return [np.uint64(mj << (31 - j)) for j, mj in enumerate(m)]


V = direction_numbers()


def sobol(i, dim):
    i = i.astype(np.uint64)
    out = np.zeros_like(i)
    for j in range(32):
        bit = (i >> np.uint64(j)) & np.uint64(1)
        out ^= bit * (np.uint64(1) << np.uint64(31 - j) if dim == 0 else V[j])
    return out


def ref_pairs(seed, gpix, pair, sample):
    g, p, s = (np.asarray(x, dtype=np.uint64) for x in np.broadcast_arrays(gpix, pair, sample))
    k0, k1 = np.uint64(seed & 0xFFFFFFFF), np.uint64(seed >> 32)
    h = hash32(np.full(g.shape, k0 ^ np.uint64(0x6a09e667), dtype=np.uint64))
    h = hash32(h ^ k1)
    h = hash32(h ^ g)
    base = hash32(h ^ p)
    i = owen(s, hash32(base))
    x = owen(sobol(i, 0), hash32(base ^ np.uint64(1)))
    y = owen(sobol(i, 1), hash32(base ^ np.uint64(2)))
    return np.stack([x, y], axis=-1).astype(np.uint32), base.astype(np.uint32)


# ------------------------------------------------------------------------------- 1. bit-exact
def test_sobol_dimension_one_from_direction_numbers_is_the_known_sequence():
    # the first 16 points of Sobol's second dimension (Joe-Kuo d = 2) in natural index order, in sixteenths:
    # V_1..V_4 = 8, 12, 10, 15 and x(i) = XOR of V_j over the set bits of i
    want = [0, 8, 12, 4, 10, 2, 6, 14, 15, 7, 3, 11, 5, 13, 9, 1]
    got = sobol(np.arange(16), 1) >> np.uint64(28)
    assert [int(x) for x in got] == want


@pytest.mark.parametrize("seed", [0, 1, 7, 0xDEADBEEFCAFEF00D])
def test_host_sampler_equals_numpy_restatement(lib, seed):
    rng = np.random.default_rng(seed & 0xFFFF)
    n = 4000
    gpix = np.concatenate([rng.integers(0, 1 << 32, n // 2, dtype=np.uint64), rng.integers(0, 1 << 24, n // 4, dtype=np.uint64),
                           np.array([0, 1, (1 << 24) - 1, 1 << 24, (1 << 32) - 1] * (n // 20), dtype=np.uint64)])[:n]
    pair = rng.integers(0, 60, n, dtype=np.uint64)
    sample = np.concatenate([rng.integers(0, 1 << 32, n // 2, dtype=np.uint64), np.arange(n // 4, dtype=np.uint64),
                             np.array([(1 << 32) - 1, (1 << 31), 0, 1, 4095] * (n // 20), dtype=np.uint64)])[:n]
    got, gbase = pairs(lib, seed, gpix, pair, sample)
    want, wbase = ref_pairs(seed, gpix, pair, sample)
    assert np.array_equal(gbase, wbase)
    assert np.array_equal(got, want)


def test_uniforms_are_the_top_24_bits_of_the_pairs(lib):
    seed, gpix, sample, depth = 0x1234_5678_9ABC, 5000, 77, 6
    u = np.zeros(5 + 2 * depth, dtype=np.float32)
    lib.hostsampler_uniforms(seed, gpix, sample, depth, u.ctypes.data)
    xy, _ = pairs(lib, seed, gpix, np.arange(3 + depth), sample)
    top = (xy >> 8).astype(np.float64) / 2.0 ** 24
    want = np.concatenate([top[0], top[1], top[2, :1], top[3:].ravel()])
    assert np.array_equal(u.astype(np.float64), want)


# ------------------------------------------------------------------------------- 2. stratification
@pytest.mark.parametrize("gpix,pair", [(0, 0), (123457, 1), (1 << 24, 2), (0xFFFFFFFF, 9), (2024, 52)])
def test_aligned_blocks_are_0k2_nets(lib, gpix, pair):
    """For k = 0..12 and blocks [m 2^k, (m + 1) 2^k), m > 0 included: for every a + b = k, each 2^-a x 2^-b box of the 24-bit
    coordinates the renderer uses holds exactly one point (so the first coordinate alone falls in 2^k distinct intervals)."""
    for k in range(13):
        for m in (0, 1, 3, (1 << (20 - k)) + 5, ((1 << 32) >> k) - 1):
            s = np.arange(m << k, (m + 1) << k, dtype=np.uint64)
            xy, _ = pairs(lib, 99, gpix, pair, s)
            q = (xy >> 8).astype(np.int64)
            for a in range(k + 1):
                b = k - a
                cell = (q[:, 0] >> (24 - a)) << b | (q[:, 1] >> (24 - b))
                assert len(np.unique(cell)) == 1 << k, (k, m, a)


# ------------------------------------------------------------------------------- 3. decorrelation
def test_first_samples_of_many_pixels_are_uniform(lib):
    xy, _ = pairs(lib, 5, np.arange(4096), 0, 0)
    u = (xy >> 8).astype(np.float64) / 2.0 ** 24
    for c in range(2):
        assert stats.kstest(u[:, c], "uniform").pvalue > 0.01


def test_pairs_of_one_pixel_are_uncorrelated(lib):
    s = np.arange(4096)
    x = [(pairs(lib, 5, 31337, p, s)[0][:, 0] >> 8).astype(np.float64) for p in (0, 1, 3)]   # camera A, camera B, bounce 1
    for i in range(3):
        for j in range(i + 1, 3):
            assert abs(np.corrcoef(x[i], x[j])[0, 1]) < 0.05, (i, j)


def test_neighbouring_pixels_get_different_point_sets(lib):
    s = np.arange(64)
    a = pairs(lib, 5, 1000, 0, s)[0]
    for g in (999, 1001, 1000 + 320):
        b = pairs(lib, 5, g, 0, s)[0]
        assert not np.array_equal(np.sort(a[:, 0]), np.sort(b[:, 0]))
        assert (a[:, 0] != b[:, 0]).mean() > 0.99
    c = pairs(lib, 6, 1000, 0, s)[0]     # and another seed moves every point
    assert (a[:, 0] != c[:, 0]).mean() > 0.99


def test_abi_flag():
    from rayz_b200 import _abi as abi
    from rayz_b200 import Backend
    assert abi.RENDER_SOBOL == 0x10
    assert Backend.params(8, 8, 1, sobol=True).flags == abi.RENDER_SOBOL
    assert Backend.params(8, 8, 1).flags == 0
    with open(os.path.join(HERE, "..", "include", "rayz_cuda.h")) as f:
        assert "#define RZ_RENDER_SOBOL 0x10u" in f.read()
    with open(os.path.join(HERE, "..", "zig", "cuda_backend.zig")) as f:
        assert "pub const RZ_RENDER_SOBOL: u32 = 0x10;" in f.read()
