"""CPU tests of the f64 path replay (oracle Scene.replay, rayz_oracle.cpp namespace replay): the backend's path algorithm
restated in f64 with the uniforms its kernels draw.

1. The replay's uniforms equal the product's bit for bit (Philox4x32-7, Owen-scrambled Sobol, the RQMC replicates and the
   pair numbers), the product side being rz_device.cuh / rz_sampler.cuh compiled as host code (tests/hostsim/sampler.cu).
2. The replay is a valid reference: in distribution it agrees with the reference restatement (Scene.render), image and
   counters, so it is not a copy of the kernel.
3. The product's f32 shading code compiled as host code (tests/hostsim/hostsim.cu: hostsim_paths) reproduces every robust
   replay path within its tolerance and with the same events, for each sampler.
4. The replay reads no product code."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

import oracle
import rayz_b200
from metrics import compare
from rayz_b200 import host
from replay_scenes import all_materials, compare_paths, config1, count_stats

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


@pytest.fixture(scope="module")
def hostsim():
    subprocess.run(["bash", os.path.join(HERE, "hostsim", "build.sh")], check=True)
    lib = C.CDLL(os.path.join(HERE, "_build", "libhostsim.so"))
    lib.hostsim_paths.argtypes = ([C.c_void_p, C.c_void_p] + [C.c_uint32] * 5 + [C.c_uint64, C.c_float, C.c_int, C.c_uint32]
                                  + [C.c_void_p] * 4)
    return lib


@pytest.fixture(scope="module")
def sampler_lib():
    subprocess.run(["bash", os.path.join(HERE, "hostsim", "build_sampler.sh")], check=True)
    lib = C.CDLL(os.path.join(HERE, "_build", "libhostsampler.so"))
    lib.hostsampler_philox.argtypes = [C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p]
    lib.hostsampler_sobol_u01.argtypes = [C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_int, C.c_void_p]
    lib.hostsampler_pair_numbers.argtypes = [C.c_uint32, C.c_void_p]
    return lib


def host_paths(lib, arrays, cam, w, h, sample_offset, spp, depth, seed, t_min=0.0, sampler="philox"):
    """hostsim_paths: the product's f32 path per (pixel, sample), shaped like Scene.replay's arrays."""
    sc, keep = host.scene_struct(arrays)
    n = (h, w, spp)
    rgb, segs = np.zeros(n + (3,), np.float32), np.zeros(n, np.uint32)
    end, hits = np.zeros(n, np.uint8), np.zeros(n + (3,), np.uint32)
    lib.hostsim_paths(C.byref(sc), C.byref(cam), w, h, sample_offset, spp, depth, seed, t_min, oracle.SAMPLERS[sampler], 0,
                      rgb.ctypes.data, segs.ctypes.data, end.ctypes.data, hits.ctypes.data)
    return dict(rgb=rgb, segs=segs, end=end, hits=hits)


# ------------------------------------------------------------------------------- 1. uniforms, bit for bit
def _u24(words):
    return (np.asarray(words, np.uint64) >> np.uint64(8)).astype(np.float64) * 2.0 ** -24


@pytest.mark.parametrize("seed", [1, 0x9E3779B97F4A7C15])
def test_replay_uniforms_equal_the_kernels(sampler_lib, seed):
    """Camera (ux, uy, ut, ur, ua) and bounce (u.x..u.w) uniforms of the replay against rz_philox / rz_sobol_u01 compiled as
    host code, with the bit layout of rz_camera_ray (high 24 bits of x, y, z, w; ua from the low bytes of x, y, z) and of
    rz_shade_segment (high 24 bits; Sobol pair 2 + s replaces u.x, u.y)."""
    depth = 6
    pairs = np.zeros(3 + depth, np.uint32)
    sampler_lib.hostsampler_pair_numbers(depth, pairs.ctypes.data)
    rng = np.random.default_rng(seed & 0xffff)
    cases = [(0, 0), (1, 1), (2**32 - 1, 2**32 - 1), (7_200_000, 4095), (123_456_789, 2**31 + 5)]
    cases += [(int(g), int(s)) for g, s in zip(rng.integers(0, 2**32, 200), rng.integers(0, 2**32, 200))]
    w = np.zeros(4, np.uint32)
    f = np.zeros(2, np.float32)
    checked = 0
    for gpix, sample in cases:
        for sampler in ("philox", "sobol", "sobol-rqmc"):
            got = oracle.replay_uniforms(seed, gpix, sample, depth, sampler)
            want = np.zeros_like(got)
            sampler_lib.hostsampler_philox(seed, gpix, sample, 0, w.ctypes.data)
            want[0:4] = _u24(w)
            want[4] = float(((int(w[0]) & 0xff) << 16) | ((int(w[1]) & 0xff) << 8) | (int(w[2]) & 0xff)) * 2.0 ** -24
            if sampler != "philox":
                rq = int(sampler == "sobol-rqmc")
                sampler_lib.hostsampler_sobol_u01(seed, gpix, int(pairs[0]), sample, rq, f.ctypes.data); want[0:2] = f
                sampler_lib.hostsampler_sobol_u01(seed, gpix, int(pairs[1]), sample, rq, f.ctypes.data); want[3:5] = f
                sampler_lib.hostsampler_sobol_u01(seed, gpix, int(pairs[2]), sample, rq, f.ctypes.data); want[2] = f[0]
            for s in range(1, depth + 1):
                sampler_lib.hostsampler_philox(seed, gpix, sample, s, w.ctypes.data)
                b = 5 + 4 * (s - 1)
                want[b:b + 4] = _u24(w)
                if sampler != "philox":
                    sampler_lib.hostsampler_sobol_u01(seed, gpix, int(pairs[2 + s]), sample, int(sampler == "sobol-rqmc"), f.ctypes.data)
                    want[b:b + 2] = f
            assert np.array_equal(got, want), (gpix, sample, sampler, np.nonzero(got != want)[0])
            checked += got.size
    assert checked > 10_000


# ------------------------------------------------------------------------------- 2. a valid reference
def test_replay_agrees_with_the_reference_in_distribution(orc):
    """Replay image vs two independently seeded Scene.render images, with the bars of
    test_hostsim_cpu.test_fp32_shading_matches_oracle_statistics; segments per path and metallic hits too.  The replay
    follows the backend's t_min = 1e-4 (the reference's is 1e-10: contact rings ~1e-4 wide, include/rayz_cuda.h), which moves
    the counters by far less than the bars."""
    t = rayz_b200.random_bouncing(128, seed=42)
    arrays, w, h, spp = t.pool.arrays(), 128, 72, 48
    sc = orc.Scene.from_arrays(arrays)
    ocam, _ = orc.default_camera(w)
    rep = sc.replay(t.camera.rz, w, h, 0, spp, 50, seed=5)
    img = rep["rgb"].mean(axis=2)
    a, st = sc.render(ocam, w, h, spp, 50, seed=11, threads=0, stats=True)
    b, _ = sc.render(ocam, w, h, spp, 50, seed=12, threads=0)
    floor, got = compare(b, a), compare(img, a)
    print("floor", floor, "\nreplay", got)
    assert got["psnr"] >= floor["psnr"] - 0.4
    assert got["block_mae"] <= floor["block_mae"] * 1.25 + 2e-4
    assert max(abs(x) for x in got["mean_diff"]) < 2.5e-3
    mine = count_stats(rep)
    paths = w * h * spp
    assert mine["ended_sky"] + mine["ended_absorbed"] + mine["ended_depth"] == paths
    assert abs(mine["segments"] / paths - st["segments"] / paths) < 0.06
    assert abs(mine["hits_metallic"] - st["hits_metallic"]) / st["hits_metallic"] < 0.03
    assert abs(mine["hits_dielectric"] - st["hits_dielectric"]) / st["hits_dielectric"] < 0.05


# ------------------------------------------------------------------------------- 3. the f32 shading code, path by path
# Fragile fractions measured on this comparison (160 x 90 or 203 x 114, 1 spp): config 1 2.7-3.1 %, glass-heavy 5.3 %, the
# all-materials scene 0.3-2.8 %; the worst robust error was 0.14 of its tolerance.  Bars: about 1.5 x the fractions.
CASES = [
    ("config1", "philox", 50, 0.0, 0.045),
    ("config1", "sobol", 50, 0.0, 0.045),
    ("config1", "sobol-rqmc", 50, 0.0, 0.045),
    ("glass", "philox", 50, 0.0, 0.08),
    ("allmat-outside", "philox", 50, 0.0, 0.04),
    ("allmat-outside", "sobol", 2, 0.0, 0.04),
    ("allmat-in_glass", "philox", 50, 1e-3, 0.04),
]


@pytest.mark.parametrize("scene,sampler,depth,t_min,fragile_max", CASES)
def test_host_f32_paths_match_the_replay(hostsim, orc, scene, sampler, depth, t_min, fragile_max):
    if scene.startswith("allmat"):
        arrays, cams, w, h = all_materials()
        cam = cams[scene.split("-")[1]]
    else:
        w, h = 160, 90
        arrays, cam = config1(w, h, glass_heavy=scene == "glass")
    off, spp = (6, 2) if sampler == "sobol-rqmc" else (3, 1)
    rep = orc.Scene.from_arrays(arrays).replay(cam, w, h, off, spp, depth, seed=7, t_min=t_min, sampler=sampler)
    got = host_paths(hostsim, arrays, cam, w, h, off, spp, depth, 7, t_min, sampler)
    compare_paths(rep, got["rgb"], f"{scene} {sampler} depth {depth}", fragile_max=fragile_max)
    rob = rep["robust"]
    for k in ("segs", "end"):
        assert np.array_equal(got[k][rob], rep[k][rob]), k
    assert np.array_equal(got["hits"][rob], rep["hits"][rob])


def test_depth_semantics_match_the_replay(hostsim, orc):
    """depth 0: every path ends at once, black, counted as ended at the depth limit; depth 1 and 2 end there."""
    arrays, cams, w, h = all_materials()
    sc = orc.Scene.from_arrays(arrays)
    for depth in (0, 1, 2):
        rep = sc.replay(cams["outside"], w, h, 0, 1, depth, seed=3)
        got = host_paths(hostsim, arrays, cams["outside"], w, h, 0, 1, depth, 3)
        compare_paths(rep, got["rgb"], f"depth {depth}")
        assert rep["segs"].max() <= max(depth, 0) and (rep["segs"][rep["end"] == oracle.END_DEPTH] == depth).all()
        if depth == 0:
            assert (rep["segs"] == 0).all() and (rep["end"] == oracle.END_DEPTH).all() and (rep["rgb"] == 0).all()
            assert (got["segs"] == 0).all() and (got["end"] == oracle.END_DEPTH).all()


# ------------------------------------------------------------------------------- 4. independence
def test_replay_reads_no_product_code():
    """The oracle stays an independent restatement (DESIGN.md section 4): it includes only standard headers, names no product
    header or source directory, does not import the product, and its Makefile adds no include path."""
    odir = os.path.join(ROOT, "oracle")
    product = re.compile(r"rayz_b200|csrc|include/|rayz_cuda|\brz_\w*\.(cuh|hpp|h)\b")
    for name in sorted(os.listdir(odir)):
        if not name.endswith((".cpp", ".hpp", ".h", ".py")) and name != "Makefile":
            continue
        text = open(os.path.join(odir, name)).read()
        for line in text.splitlines():
            if re.match(r"\s*#\s*include", line):
                assert re.match(r"\s*#\s*include\s*<\w+>\s*$", line), f"{name}: {line.strip()}"
                assert not product.search(line), f"{name}: {line.strip()}"
            assert not re.match(r"\s*(import|from)\s+(rayz_b200|host)\b", line), f"{name}: {line.strip()}"
        if name == "Makefile":
            assert not re.search(r"(^|\s)-(I|isystem|iquote|include)", text), "oracle/Makefile adds an include path"
            assert not product.search(text), "oracle/Makefile names product sources"
