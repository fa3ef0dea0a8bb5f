"""GPU parity tests: the CUDA backend (through the C ABI) against the CPU oracle.

All tests here need a B200 (`-m gpu`).  Bars (SURVEY.md §8c / BASELINE.json north_star):
  * primary-ray closest-hit sphere ids: BIT-EXACT against the oracle and the committed goldens;
  * converged images: within the Monte-Carlo noise floor of the oracle itself.  The reference's
    sequential PRNG cannot be matched sample for sample, so the comparison is statistical: with
    per-pixel variance s2 ~= 0.027 the MSE between two independent N-spp renders is ~ s2*(2/N).
    Stated tolerance at 500 vs 500 spp (config 2): linear PSNR >= 38 dB, per-channel MAE <= 0.008,
    |global mean difference| <= 5e-4 per channel, 16x16 block-mean MAE <= 0.002.  At other spp the
    floor is MEASURED with a second, independently seeded oracle render and the GPU image must be
    within 0.3 dB / 5 % of it.
"""
import os

import numpy as np
import pytest

import rayz_b200
from rayz_b200 import Backend
from rayz_b200 import _abi as abi
from metrics import compare

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def be():
    b = Backend((0,))
    yield b
    b.close()


@pytest.fixture(scope="module")
def scene42():
    return rayz_b200.random_bouncing(400, seed=42).pool.arrays()


def cam_for(w):
    h = int(w / rayz_b200.ASPECT_RATIO)
    return rayz_b200.Camera.init(20.0, 10.0, 0.6, (13, 2, 3), (0, 0, 0), (0, 1, 0), h, w).rz, h


def fnv1a(a: np.ndarray) -> int:
    h = 0xcbf29ce484222325
    for b in np.ascontiguousarray(a).view(np.uint8).tobytes()[::97]:  # strided: keeps the python loop short
        h = ((h ^ b) * 0x100000001b3) & 0xFFFFFFFFFFFFFFFF
    return h


# ------------------------------------------------------------------------------- K0: ids, bit-exact
@pytest.mark.parametrize("w", [400, 1200])
def test_primary_ids_bit_exact_default_scene(be, scene42, orc, w):
    be.upload_scene(scene42)
    cam, h = cam_for(w)
    ids_bvh = be.primary_ids(cam, w, h, use_bvh=True)
    ids_bf = be.primary_ids(cam, w, h, use_bvh=False)
    gold = np.load(os.path.join(GOLDEN, f"ids_seed42_{w}x{h}.npz"))["ids"].astype(np.int32)
    assert np.array_equal(ids_bvh, gold), f"{(ids_bvh != gold).sum()} of {gold.size} ids differ from the golden fixture"
    assert np.array_equal(ids_bf, gold)
    assert fnv1a(ids_bvh) == fnv1a(gold)
    ocam, oh = orc.default_camera(w)
    ref = orc.Scene.from_arrays(scene42).primary_ids(ocam, w, oh)
    assert np.array_equal(ids_bvh, ref)


@pytest.mark.parametrize("kw", [dict(seed=7), dict(seed=42, glass_heavy=True), dict(seed=3, grid_lo=-30, grid_hi=30)])
def test_primary_ids_bit_exact_other_scenes(be, orc, kw):
    arrays = rayz_b200.random_bouncing(320, **kw).pool.arrays()
    be.upload_scene(arrays)
    cam, h = cam_for(320)
    ocam, _ = orc.default_camera(320)
    ref = orc.Scene.from_arrays(arrays).primary_ids(ocam, 320, h)
    assert np.array_equal(be.primary_ids(cam, 320, h, use_bvh=True), ref)
    assert np.array_equal(be.primary_ids(cam, 320, h, use_bvh=False), ref)


def _tiny_pool(n, moving=False):
    rng = np.random.default_rng(5 + n)
    pool = rayz_b200.MemPool()
    t = pool.add_solid((0.5, 0.5, 0.5))
    for i in range(n):
        c = rng.uniform(-2, 2, 3)
        v = rng.uniform(-0.5, 0.5, 3) if (moving and i % 2) else (0, 0, 0)
        pool.add_sphere(c, float(rng.uniform(0.2, 0.9)), pool.add_diffuse(t), v)
    return pool.arrays()


@pytest.mark.parametrize("n,moving", [(1, False), (2, False), (3, True), (5, True), (64, True)])
def test_primary_ids_small_scenes_and_camera_inside(be, orc, n, moving):
    arrays = _tiny_pool(n, moving)
    be.upload_scene(arrays)
    osc = orc.Scene.from_arrays(arrays)
    for look_from in ((0, 0, 6), (0.1, 0.0, 0.2)):   # outside, and (likely) inside a sphere
        cam = rayz_b200.Camera.init(60.0, 5.0, 0.0, look_from, (0, 0, 0), (0, 1, 0), 48, 64).rz
        ocam = orc.camera(60.0, 5.0, 0.0, look_from, (0, 0, 0), (0, 1, 0), 48, 64)
        ref = osc.primary_ids(ocam, 64, 48)
        assert np.array_equal(be.primary_ids(cam, 64, 48, True), ref)
        assert np.array_equal(be.primary_ids(cam, 64, 48, False), ref)


# ------------------------------------------------------------------------------- K1: converged image
def _oracle_pair(orc, arrays, w, h, spp, depth=50):
    sc = orc.Scene.from_arrays(arrays)
    ocam, oh = orc.default_camera(w)
    assert oh == h
    a, st = sc.render(ocam, w, h, spp, depth, seed=101, threads=0, stats=True)
    b, _ = sc.render(ocam, w, h, spp, depth, seed=202, threads=0)
    return a, b, st


@pytest.mark.parametrize("variant", ["mega", "bvh"])
def test_image_parity_default_scene(be, scene42, orc, variant):
    """Config-1 size (400x225), 128 spp: GPU image vs oracle within the measured noise floor."""
    w, spp = 400, 128
    cam, h = cam_for(w)
    be.upload_scene(scene42)
    lin, rgb8, n = be.render(cam, Backend.params(w, h, spp, 50, seed=1, variant=variant, collect_stats=True))
    assert n == w * h * spp
    assert np.isfinite(lin).all() and (lin[..., 3] == 1).all()
    gst = be.stats()
    a, b, ost = _oracle_pair(orc, scene42, w, h, spp)
    floor = compare(b, a)
    got = compare(lin[..., :3], a)
    print("floor", floor, "\ngpu  ", got)
    assert got["psnr"] >= floor["psnr"] - 0.3
    assert max(got["mae"]) <= max(floor["mae"]) * 1.05
    assert got["block_mae"] <= floor["block_mae"] * 1.15 + 1e-4
    sigma = (0.027 * 2 / (spp * w * h)) ** 0.5 * 3.0   # channels/pixels are correlated: x3
    assert max(abs(x) for x in got["mean_diff"]) <= max(5e-4, 4 * sigma)
    # path statistics (SURVEY probe: 2.756 seg/path, 99.9 % end on the sky).  The reference traps
    # ~0.04 % of paths inside spheres through t~1e-10 self-hits (DESIGN.md "known deviation"),
    # which shows up as ended_depth and ~1 % more diffuse hits on its side only.
    gs, os_ = gst["segments"] / gst["paths"], ost["segments"] / ost["paths"]
    assert gst["paths"] == n and abs(gs - os_) / os_ < 0.012
    assert abs(gst["ended_sky"] / n - ost["ended_sky"] / n) < 1.5e-3
    assert abs(gst["hits_metallic"] - ost["hits_metallic"]) / ost["hits_metallic"] < 0.01
    assert abs(gst["hits_dielectric"] - ost["hits_dielectric"]) / ost["hits_dielectric"] < 0.015
    assert gst["ended_sky"] + gst["ended_absorbed"] + gst["ended_depth"] == gst["paths"]


def test_image_parity_config2_against_golden_blocks(be, scene42):
    """Config 2 at full size and spp (1200x675, 500 spp) vs the committed oracle block means."""
    path = os.path.join(GOLDEN, "config2_oracle_500spp.npz")
    if not os.path.exists(path):
        pytest.skip("golden block means not generated")
    g = np.load(path)
    w, spp = 1200, 500
    cam, h = cam_for(w)
    be.upload_scene(scene42)
    lin, _, n = be.render(cam, Backend.params(w, h, spp, 50, seed=1, variant="auto"), want_rgb8=False)
    img = lin[..., :3].astype(np.float64)
    blk = lambda x, b: x[:h // b * b, :w // b * b].reshape(h // b, b, w // b, b, 3).mean(axis=(1, 3))
    d_mean = img.mean(axis=(0, 1)) - g["mean"]
    b16 = np.abs(blk(img, 16) - g["block16"]).mean()
    b4 = blk(img, 4) - g["block4"]
    psnr4 = 10 * np.log10(1.0 / (b4 * b4).mean())
    print("mean diff", d_mean, "block16 mae", b16, "block4 psnr", psnr4)
    assert np.abs(d_mean).max() <= 5e-4
    assert b16 <= 0.002
    # 4x4 block means average 16 pixels: floor ~ 39.7 dB + 10log10(16) ~ 51.7 dB at 500 vs 500 spp
    assert psnr4 >= 49.0
    # per pixel, at the committed sample of the same oracle render (its 16x16 block MAE is b16 above)
    px = np.load(os.path.join(GOLDEN, "config2_oracle_500spp_pixels.npz"))
    got = compare(img.reshape(-1, 1, 3)[px["idx"]], px["rgb"][:, None])
    print("full-res pixel sample", got)
    assert got["psnr"] >= 38.0 and max(got["mae"]) <= 0.008


def test_glass_heavy_scene_parity(be, orc):
    """Config 5 scene (all-dielectric): long paths, total internal reflection, depth limit."""
    arrays = rayz_b200.random_bouncing(320, seed=42, glass_heavy=True).pool.arrays()
    w, spp = 320, 96
    cam, h = cam_for(w)
    be.upload_scene(arrays)
    lin, _, n = be.render(cam, Backend.params(w, h, spp, 50, seed=3, variant="mega", collect_stats=True))
    gst = be.stats()
    a, b, ost = _oracle_pair(orc, arrays, w, h, spp)
    floor, got = compare(b, a), compare(lin[..., :3], a)
    print("floor", floor, "\ngpu  ", got, "\n", gst, "\n", ost)
    assert got["psnr"] >= floor["psnr"] - 0.3 and got["block_mae"] <= floor["block_mae"] * 1.15 + 1e-4
    assert max(abs(x) for x in got["mean_diff"]) <= 1e-3
    assert abs(gst["segments"] / n - ost["segments"] / n) / (ost["segments"] / n) < 0.02


def test_moving_spheres_and_all_materials_small_scene(be, orc):
    """Hand-built scene: moving diffuse, fuzzy metal, glass + hollow glass, checker ground, all three diffuse methods."""
    pool = rayz_b200.MemPool()
    ck = pool.add_checker(0.5, pool.add_solid((0.1, 0.2, 0.6)), pool.add_solid((0.9, 0.9, 0.8)))
    pool.add_sphere((0, -100.5, -1), 100, pool.add_diffuse(ck))
    pool.add_sphere((0, 0, -1.2), 0.5, pool.add_diffuse(pool.add_solid((0.7, 0.3, 0.3)), abi.DIFFUSE_UNIT_SPHERE_SURFACE), (0, 0.4, 0))
    pool.add_sphere((-1, 0, -1), 0.5, pool.add_dielectric(1.5))
    pool.add_sphere((-1, 0, -1), 0.4, pool.add_dielectric(1.0 / 1.5))       # hollow bubble (penultimateScene)
    pool.add_sphere((1, 0, -1), 0.5, pool.add_metallic(pool.add_solid((0.8, 0.6, 0.2)), 0.7))
    pool.add_sphere((0.3, 0.9, -1.5), 0.35, pool.add_diffuse(pool.add_solid((0.2, 0.8, 0.3)), abi.DIFFUSE_UNIT_SPHERE), (0.5, 0, 0))
    pool.add_sphere((2.0, 0.2, -2.5), 0.7, pool.add_metallic(pool.add_solid((0.9, 0.9, 0.9)), 0.0))
    arrays = pool.arrays()
    w, h, spp = 256, 144, 128
    args = (30.0, 3.4, 2.0, (-2, 2, 1), (0, 0, -1), (0, 1, 0), h, w)
    cam, ocam = rayz_b200.Camera.init(*args).rz, orc.camera(*args)
    be.upload_scene(arrays)
    osc = orc.Scene.from_arrays(arrays)
    assert np.array_equal(be.primary_ids(cam, w, h), osc.primary_ids(ocam, w, h))
    a, _ = osc.render(ocam, w, h, spp, 50, seed=1, threads=0)
    b, _ = osc.render(ocam, w, h, spp, 50, seed=2, threads=0)
    floor = compare(b, a)
    for variant in ("mega", "bvh"):
        lin, _, _ = be.render(cam, Backend.params(w, h, spp, 50, seed=9, variant=variant))
        got = compare(lin[..., :3], a)
        print(variant, "floor", floor, "\ngpu  ", got)
        assert got["psnr"] >= floor["psnr"] - 0.3 and got["block_mae"] <= floor["block_mae"] * 1.2 + 1e-4
        assert max(abs(x) for x in got["mean_diff"]) <= 1.5e-3


# ------------------------------------------------------------------------------- invariances
def test_sharding_and_tuning_are_bit_identical(be, scene42):
    """Counter-based RNG + integer accumulation: any row sharding / work-unit size / rays-per-thread
    reproduces the full-frame image bit for bit (this is what makes multi-GPU slabs exact)."""
    w, spp = 200, 24
    cam, h = cam_for(w)
    be.upload_scene(scene42)
    be.set_tuning(2, 16)
    full_lin, full_rgb, _ = be.render(cam, Backend.params(w, h, spp, 50, seed=77, variant="mega"))
    for count, band in ((2, 4), (3, 1), (8, 4)):
        lin = np.empty_like(full_lin); rgb = np.empty_like(full_rgb)
        for s in range(count):
            p = Backend.params(w, h, spp, 50, seed=77, variant="mega", shard_index=s, shard_count=count, band_rows=band)
            l, r, n = be.render(cam, p)
            rows = [j for j in range(h) if (j // band) % count == s]
            assert l.shape[0] == len(rows) and n == len(rows) * w * spp
            lin[rows] = l; rgb[rows] = r
        assert np.array_equal(lin, full_lin) and np.array_equal(rgb, full_rgb)
    for rpt, chunk in ((1, 16), (2, 5), (1, 64)):
        be.set_tuning(rpt, chunk)
        l, r, _ = be.render(cam, Backend.params(w, h, spp, 50, seed=77, variant="mega"))
        assert np.array_equal(l, full_lin) and np.array_equal(r, full_rgb), (rpt, chunk)
    be.set_tuning(2, 16)
    # a different seed must change the image
    l2, _, _ = be.render(cam, Backend.params(w, h, spp, 50, seed=78, variant="mega"))
    assert not np.array_equal(l2, full_lin)


def test_bvh_variant_matches_brute_force(be, scene42):
    """Same RNG keys, same closest hit => the BVH kernel reproduces the brute-force image except where
    FP32 search order breaks a near-tie (a handful of samples)."""
    w, spp = 200, 16
    cam, h = cam_for(w)
    be.upload_scene(scene42)
    a, _, _ = be.render(cam, Backend.params(w, h, spp, 50, seed=5, variant="mega"))
    b, _, _ = be.render(cam, Backend.params(w, h, spp, 50, seed=5, variant="bvh"))
    same = (a == b).all(axis=-1).mean()
    print("pixels bit-identical:", same)
    assert same > 0.995
    assert compare(a[..., :3], b[..., :3])["psnr"] > 45


def test_progressive_accumulation_sample_offset(be, scene42):
    w, spp = 160, 8
    cam, h = cam_for(w)
    be.upload_scene(scene42)
    a, _, _ = be.render(cam, Backend.params(w, h, spp, 50, seed=4, sample_offset=0))
    b, _, _ = be.render(cam, Backend.params(w, h, spp, 50, seed=4, sample_offset=spp))
    c, _, _ = be.render(cam, Backend.params(w, h, 2 * spp, 50, seed=4))
    assert np.abs((a.astype(np.float64) + b) / 2 - c).max() < 1e-6


# ------------------------------------------------------------------------------- K5 + edges + errors
def test_quantise_matches_writeppm_transform(be, scene42, orc):
    w, spp = 240, 16
    cam, h = cam_for(w)
    be.upload_scene(scene42)
    lin, rgb8, _ = be.render(cam, Backend.params(w, h, spp, 50, seed=2))
    ref = orc.quantise(lin[..., :3].astype(np.float64))
    d = np.abs(ref.astype(np.int32) - rgb8.astype(np.int32))
    # the device quantises the f64 mean, the check re-quantises its float32 rounding: <= 1 LSB on a few pixels
    assert d.max() <= 1 and (d != 0).mean() < 2e-3


@pytest.mark.parametrize("w,h,spp,depth", [(1, 1, 1, 50), (33, 19, 3, 50), (64, 36, 7, 1), (64, 36, 4, 0), (31, 5, 17, 2)])
def test_edge_sizes(be, scene42, w, h, spp, depth):
    be.upload_scene(scene42)
    cam = rayz_b200.Camera.init(20.0, 10.0, 0.6, (13, 2, 3), (0, 0, 0), (0, 1, 0), h, w).rz
    for variant in ("mega", "bvh"):
        lin, rgb8, n = be.render(cam, Backend.params(w, h, spp, depth, seed=1, variant=variant, collect_stats=True))
        st = be.stats()
        assert n == w * h * spp == st["paths"]
        assert lin.shape == (h, w, 4) and np.isfinite(lin).all()
        if depth == 0:
            assert (lin[..., :3] == 0).all() and st["segments"] == 0 and st["ended_depth"] == n   # renderer.zig:104-105
        else:
            assert st["segments"] >= n and (lin[..., :3] >= 0).all() and (lin[..., :3] <= 1.0 + 1e-6).all()
        if depth == 1:
            assert st["segments"] == n   # exactly one closest-hit query per path


def test_single_sphere_scene_and_sky(be, orc):
    pool = rayz_b200.MemPool()
    pool.add_sphere((0, 0, -3), 1.0, pool.add_diffuse(pool.add_solid((0.5, 0.5, 0.5))))
    be.upload_scene(pool.arrays())
    args = (40.0, 3.0, 0.0, (0, 0, 0), (0, 0, -1), (0, 1, 0), 40, 40)
    cam = rayz_b200.Camera.init(*args).rz
    lin, _, _ = be.render(cam, Backend.params(40, 40, 64, 50, seed=1))
    # a corner pixel sees only sky: ((1-t)+c)*t with t = (unit(dir).y+1)/2   (renderer.zig:124-125)
    ocam = orc.camera(*args)
    o, d, _ = orc.get_ray(ocam, 0, 0)
    t = 0.5 * (d[1] / np.linalg.norm(d) + 1)
    want = np.array([(1 - t + 0.5) * t, (1 - t + 0.7) * t, (1 - t + 1.0) * t])
    assert np.allclose(lin[0, 0, :3], want, atol=5e-3)
    assert lin[20, 20, :3].max() < want.max()   # centre pixel is on the grey sphere: darker than sky


def test_error_behaviour(be, scene42):
    fresh = Backend((0,))
    cam, h = cam_for(64)
    with pytest.raises(abi.BackendError) as e:
        fresh.render(cam, Backend.params(64, h, 1))
    assert e.value.code == -6                                  # RZ_ERR_NO_SCENE
    with pytest.raises(abi.BackendError):
        fresh.primary_ids(cam, 64, h)
    fresh.upload_scene(scene42)
    with pytest.raises(abi.BackendError) as e:
        fresh.render(cam, Backend.params(64, h, 1, variant=9))
    assert e.value.code == -1
    with pytest.raises(abi.BackendError):
        fresh.render(cam, Backend.params(64, h, 0))
    with pytest.raises(abi.BackendError):
        fresh.render(cam, Backend.params(64, h, 1, shard_index=2, shard_count=2))
    bad = dict(scene42); bad["sphere_material"] = scene42["sphere_material"].copy(); bad["sphere_material"][3] = 10 ** 6
    with pytest.raises(abi.BackendError):
        fresh.upload_scene(bad)
    with pytest.raises(abi.BackendError):
        Backend((99,))
    fresh.close()


def test_tracer_render_is_a_drop_in(orc):
    """The reference's call sequence (rayz.zig:22-41): build scene, render(), use img."""
    tracer = rayz_b200.random_bouncing(160, seed=42)
    assert tracer.samples_per_px == 10 and tracer.max_bounces == 50
    rays = tracer.render()
    assert rays == 160 * 90 * 10                                # renderer.zig:90,100
    img = tracer.img.pixels.reshape(90, 160, 3)
    sc = orc.Scene.from_arrays(tracer.pool.arrays())
    ocam, _ = orc.default_camera(160)
    ref, _ = sc.render(ocam, 160, 90, 10, 50, seed=1, threads=0)
    assert np.abs(img.mean(axis=(0, 1)) - ref.mean(axis=(0, 1))).max() < 6e-3
    import io
    buf = io.StringIO()
    tracer.img.writePPM(buf)
    lines = buf.getvalue().split("\n")
    assert lines[:3] == ["P3", "160 90", "255"] and len(lines) == 3 + 160 * 90 + 1
    assert lines[3] == " ".join(str(int(x)) for x in tracer.img.rgb8[0, 0])


def test_fp32_peak_microbenchmark_is_sane(be):
    tf, sms = be.fp32_peak(100)
    assert sms >= 100 and 30.0 < tf < 90.0, (tf, sms)


def test_wavefront_matches_megakernel_bitwise(be, scene42):
    """K2 (staged kernels, ballot compaction, CUDA graph) runs the same search/shade functions with the
    same RNG keys as K1, and accumulation is integer: the images must be bit-identical."""
    w, spp = 200, 12
    cam, h = cam_for(w)
    be.upload_scene(scene42)
    a, a8, _ = be.render(cam, Backend.params(w, h, spp, 50, seed=21, variant="mega", collect_stats=True))
    sa = be.stats()
    b, b8, n = be.render(cam, Backend.params(w, h, spp, 50, seed=21, variant="wavefront", collect_stats=True))
    sb = be.stats()
    assert n == w * h * spp
    assert np.array_equal(a, b) and np.array_equal(a8, b8)
    for k in ("paths", "segments", "hits_diffuse", "hits_metallic", "hits_dielectric", "ended_sky", "ended_absorbed", "ended_depth"):
        assert sa[k] == sb[k], k
    # edge: sizes that leave padding pixels and a depth-0 render
    for (ww, hh, s, d) in ((33, 19, 3, 50), (16, 9, 2, 0)):
        c2 = rayz_b200.Camera.init(20.0, 10.0, 0.6, (13, 2, 3), (0, 0, 0), (0, 1, 0), hh, ww).rz
        x, _, _ = be.render(c2, Backend.params(ww, hh, s, d, seed=3, variant="mega"))
        y, _, _ = be.render(c2, Backend.params(ww, hh, s, d, seed=3, variant="wavefront"))
        assert np.array_equal(x, y)


def _n_gpus():
    import torch
    return torch.cuda.device_count()


@pytest.mark.skipif("_n_gpus() < 2")
def test_multi_device_context_matches_single_device_bitwise(scene42):
    """One process driving N GPUs (RzConfig.n_devices): rows are dealt in bands, each device's resolve
    kernel writes straight into GPU0's framebuffer over NVLink P2P.  Must equal the 1-GPU render bit for bit."""
    n = min(_n_gpus(), 4)
    w, spp = 320, 16
    cam, h = cam_for(w)
    one = Backend((0,))
    one.upload_scene(scene42)
    a, a8, na = one.render(cam, Backend.params(w, h, spp, 50, seed=31, variant="mega"))
    many = Backend(tuple(range(n)))
    many.upload_scene(scene42)
    for variant in ("mega", "bvh"):
        b, b8, nb = many.render(cam, Backend.params(w, h, spp, 50, seed=31, variant=variant, collect_stats=True))
        assert na == nb == w * h * spp == many.stats()["paths"]
        if variant == "mega":
            assert np.array_equal(a, b) and np.array_equal(a8, b8)
        else:   # another kernel family: equal up to the FP32-test-vs-exact-box edge (see test_staged_cull_is_conservative...)
            assert int((a != b).any(axis=-1).sum()) <= 2
    # a multi-device context that is itself one shard of a larger job
    full = np.empty_like(a)
    for s in range(2):
        l, _, _ = many.render(cam, Backend.params(w, h, spp, 50, seed=31, variant="mega", shard_index=s, shard_count=2, band_rows=4))
        # context shard s of 2 with n devices == shards s*n..s*n+n-1 of 2n
        rows = sorted(j for d in range(n) for j in range(h) if (j // 4) % (2 * n) == s * n + d)
        assert l.shape[0] == len(rows)
        full[rows] = l
    assert np.array_equal(full, a)
    # page-locked host buffers: no gather at all, every device copies its own bands into the caller's frame (one strided
    # cudaMemcpy2DAsync per device and buffer) — same bytes; sizes whose last band is partial (90 = 22 bands of 4 + 2 rows)
    import torch
    for ww, sc in ((w, 1), (160, 1), (w, 2)):
        cam2, hh = cam_for(ww)
        ref_l, ref_8, _ = one.render(cam2, Backend.params(ww, hh, spp, 50, seed=31, variant="mega"))
        for s_ in range(sc):
            pp = Backend.params(ww, hh, spp, 50, seed=31, variant="mega", shard_index=s_, shard_count=sc, band_rows=4)
            rows = many.shard_rows(pp)
            pl = torch.empty((rows, ww, 4), dtype=torch.float32).pin_memory().numpy()
            p8 = torch.empty((rows, ww, 3), dtype=torch.uint8).pin_memory().numpy()
            pl[:] = -1; p8[:] = 7
            many.render(cam2, pp, out_linear=pl, out_rgb8=p8)
            want = list(range(hh)) if sc == 1 else sorted(j for d in range(n) for j in range(hh) if (j // 4) % (sc * n) == s_ * n + d)
            assert np.array_equal(pl, ref_l[want]) and np.array_equal(p8, ref_8[want]), (ww, sc, s_)
    one.close(); many.close()


# ---------------------------------------------------------------------------------------------
# K4: device LBVH build (rz_bvh_build.cu).  Closest hits do not depend on the tree, so an image
# traced through the device-built tree must equal the host-SAH one (and the brute-force one) bit
# for bit; primary ids through the lazily built reference-shaped tree are unchanged.
# ---------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_device_lbvh_matches_host_sah_and_bruteforce_bitwise(scene42):
    w, spp = 240, 8
    cam, h = cam_for(w)
    host = Backend((0,), bvh_build="host")
    host.upload_scene(scene42)
    dev = Backend((0,), bvh_build="device")
    dev.upload_scene(scene42)
    assert dev.timing()["bvh_build_us"] > 0
    a, a8, _ = host.render(cam, Backend.params(w, h, spp, 50, seed=9, variant="bvh"))
    b, b8, _ = dev.render(cam, Backend.params(w, h, spp, 50, seed=9, variant="bvh", collect_stats=True))
    st = dev.stats()
    m, m8, _ = dev.render(cam, Backend.params(w, h, spp, 50, seed=9, variant="mega"))
    assert np.array_equal(a, b) and np.array_equal(a8, b8)      # two trees, the same sphere tests: bit for bit
    assert int((m != b).any(axis=-1).sum()) <= 2                # brute force vs BVH: up to the documented FP32 edge
    assert st["node_tests"] > 0 and st["sphere_tests"] > 0
    ids_h = host.primary_ids(cam, w, h, use_bvh=True)
    ids_d = dev.primary_ids(cam, w, h, use_bvh=True)
    assert np.array_equal(ids_h, ids_d)
    # the LBVH's leaf size (RzTuning::lbvh_leaf; default 1) shapes the tree, never the image: fewer, fuller leaves test more spheres
    tests_per_leaf = {}
    for leaf in (1, 4, 8):
        dl = Backend((0,), bvh_build="device")
        dl.set_tuning(lbvh_leaf=leaf)                            # (applies at the upload)
        dl.upload_scene(scene42)
        c, c8, _ = dl.render(cam, Backend.params(w, h, spp, 50, seed=9, variant="bvh", collect_stats=True))
        assert np.array_equal(a, c) and np.array_equal(a8, c8), leaf
        tests_per_leaf[leaf] = dl.stats()["sphere_tests"]
        dl.close()
    assert tests_per_leaf[1] < tests_per_leaf[4] < tests_per_leaf[8]


@pytest.mark.gpu
@pytest.mark.parametrize("n_spheres", [1, 2, 3, 5, 33])
def test_device_lbvh_tiny_scenes(n_spheres):
    """Degenerate trees: one sphere (no internal node), two, odd counts, duplicate centres (equal Morton codes)."""
    rng = np.random.default_rng(n_spheres)
    pool = rayz_b200.MemPool()
    t = pool.add_solid((0.5, 0.6, 0.7))
    centres = rng.uniform(-2, 2, size=(n_spheres, 3))
    if n_spheres >= 3:
        centres[2] = centres[1]          # identical centre => identical Morton code, tie broken by index
    for i in range(n_spheres):
        v = rng.uniform(-0.4, 0.4, 3) if i % 2 else (0, 0, 0)
        pool.add_sphere(centres[i], 0.5 + 0.1 * (i % 3), pool.add_diffuse(t), v)
    scene = pool.arrays()
    cam = rayz_b200.Camera.init(60.0, 6.0, 0.0, (0, 0, 6), (0, 0, 0), (0, 1, 0), 48, 64).rz
    host = Backend((0,), bvh_build="host")
    host.upload_scene(scene)
    dev = Backend((0,), bvh_build="device")
    dev.upload_scene(scene)
    a, _, _ = host.render(cam, Backend.params(64, 48, 16, 8, seed=3, variant="bvh"))
    b, _, _ = dev.render(cam, Backend.params(64, 48, 16, 8, seed=3, variant="bvh"))
    m, _, _ = dev.render(cam, Backend.params(64, 48, 16, 8, seed=3, variant="mega"))
    assert np.array_equal(a, b) and int((m != b).any(axis=-1).sum()) <= 2
    assert float(b[..., :3].max()) > 0


@pytest.mark.gpu
def test_device_lbvh_100k_spheres_config4():
    """BASELINE config 4 geometry (99,856 spheres): device LBVH vs host SAH, bit-identical image; build times reported."""
    t = rayz_b200.random_bouncing(320, seed=42, grid_lo=-158, grid_hi=158)
    scene = t.pool.arrays()
    assert len(scene["sphere_radius"]) > 99000
    host = Backend((0,), bvh_build="host")
    host.upload_scene(scene)
    dev = Backend((0,))                  # auto: >= 8192 spheres => device build
    dev.upload_scene(scene)
    th, td = host.timing()["bvh_build_us"], dev.timing()["bvh_build_us"]
    print(f"\n100k-sphere BVH build: host SAH {th / 1e3:.1f} ms, device LBVH {td / 1e3:.3f} ms")
    assert 0 < td < th
    p = Backend.params(t.img.w, t.img.h, 4, 50, seed=2, variant="auto", collect_stats=True)
    a, _, _ = host.render(t.camera.rz, p)
    sh = host.stats()
    b, _, _ = dev.render(t.camera.rz, p)
    sd = dev.stats()
    assert host.timing()["variant"] == 3 and dev.timing()["variant"] == 3
    # Not bit-identical at this scale, by a hair: 200 units away the FP32 discriminant |oc|^2 - r^2 carries an absolute
    # error of ~2e-3 against r^2 = 0.04, so a grazing ray can "hit" a sphere a few 1e-3 outside its box; whether that
    # sphere is tested then depends on how the tree groups it (brute force always tests it).  Measured: 1 pixel of
    # 57,600 (230k paths).  The 485-sphere scene, where rays stay within ~30 units, is bit-identical (tests above).
    n_diff = int((a != b).any(axis=-1).sum())
    print(f"pixels differing between the two trees: {n_diff} of {a.shape[0] * a.shape[1]}")
    assert n_diff <= 6
    assert float(np.abs(a - b).mean()) < 1e-5
    print(f"node tests/segment: SAH {sh['node_tests'] / sh['segments']:.1f}, LBVH {sd['node_tests'] / sd['segments']:.1f}; "
          f"sphere tests/segment: SAH {sh['sphere_tests'] / sh['segments']:.2f}, LBVH {sd['sphere_tests'] / sd['segments']:.2f}")


# ---------------------------------------------------------------------------------------------
# Staged K1 (primary kernel -> sorted stages -> persistent megakernel).  Culling only ever removes
# spheres a ray cannot hit, so every form must equal the single persistent kernel bit for bit.
# ---------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("tail", ["bvh", "brute"])
def test_staged_megakernel_equals_single_kernel_bitwise_and_stage_stats(scene42, tail):
    """tail = which kernel takes the paths after the sorted stages: the BVH kernel (default) or the brute-force megakernel."""
    be = Backend((0,))
    be.set_tuning(tail_brute=int(tail == "brute"))
    w, spp = 320, 24
    cam, h = cam_for(w)
    be.upload_scene(scene42)
    a, a8, na = be.render(cam, Backend.params(w, h, spp, 50, seed=5, variant="mega_single", collect_stats=True))
    s1 = be.stats()
    assert be.timing()["variant"] == 4 and be.timing()["passes"] == 0
    b, b8, nb = be.render(cam, Backend.params(w, h, spp, 50, seed=5, variant="mega", collect_stats=True))
    s2 = be.stats()
    st = [be.stage_stats(k) for k in range(3)]
    assert be.timing()["variant"] == 1 and be.timing()["passes"] >= 1
    assert np.array_equal(a, b) and np.array_equal(a8, b8) and na == nb
    n = len(scene42["sphere_radius"])
    for k in ("paths", "segments", "ended_sky", "ended_absorbed", "ended_depth", "hits_diffuse", "hits_metallic", "hits_dielectric"):
        assert s1[k] == s2[k], k
        assert sum(s[k] for s in st) == s2[k], k
    assert s1["sphere_tests"] == s1["segments"] * n                    # brute force tests everything
    assert st[0]["segments"] == s2["paths"] and st[0]["paths"] == s2["paths"]   # one camera segment per path
    if tail == "brute":
        assert st[2]["sphere_tests"] == st[2]["segments"] * n and st[2]["node_tests"] == 0   # the persistent stage is brute force too
    else:
        assert 0 < st[2]["sphere_tests"] < 0.05 * st[2]["segments"] * n and st[2]["node_tests"] > st[2]["segments"]   # it walked the tree
    assert st[0]["node_tests"] == 0 and st[1]["node_tests"] == 0
    assert st[0]["sphere_tests"] < 0.15 * st[0]["segments"] * n        # tile-frustum cull
    assert st[1]["sphere_tests"] < 0.50 * st[1]["segments"] * n        # sorted-unit cull
    assert s2["sphere_tests"] < 0.4 * s1["sphere_tests"]
    c, _, _ = be.render(cam, Backend.params(w, h, spp, 50, seed=5, variant="mega", serial_passes=True))
    assert np.array_equal(a, c)
    for ue in (64, 1024, 2048):                     # entries per sorted-stage work unit: only the cull's grain changes
        be.set_tuning(unit_entries=ue)
        d, _, _ = be.render(cam, Backend.params(w, h, spp, 50, seed=5, variant="mega"))
        assert np.array_equal(a, d), ue
    be.set_tuning(unit_entries=512)
    for sectors in (0, 1, 2):                       # direction field of the sort key: octants, 45- or 22.5-degree sectors (default: by the box's shape)
        for stages in (1, 3, 8):                    # and the number of sorted stages: the culls never change a closest hit
            be.set_tuning(key_sectors=sectors, second_stages=stages)
            d, _, _ = be.render(cam, Backend.params(w, h, spp, 50, seed=5, variant="mega"))
            assert np.array_equal(a, d), (sectors, stages)
    be.close()


@pytest.mark.gpu
def test_staged_megakernel_many_small_passes(be, scene42):
    """A tiny queue (2^16 entries) forces dozens of passes over both streams; the image must not change."""
    w, spp = 256, 32
    cam, h = cam_for(w)
    be.upload_scene(scene42)
    ref, _, _ = be.render(cam, Backend.params(w, h, spp, 50, seed=11, variant="mega_single"))
    fresh = Backend((0,))               # buffers are sized at the first render of a context
    fresh.set_tuning(queue_log2=16)
    fresh.upload_scene(scene42)
    out, _, _ = fresh.render(cam, Backend.params(w, h, spp, 50, seed=11, variant="mega"))
    assert fresh.timing()["passes"] > 8
    assert np.array_equal(ref, out)
    out2, _, _ = fresh.render(cam, Backend.params(w, h, spp, 50, seed=11, variant="mega", serial_passes=True))
    assert np.array_equal(ref, out2)
    for stages, tail in ((0, "bvh"), (1, "brute"), (5, "bvh"), (4, "brute"), (8, "bvh")):
        fresh.set_tuning(second_stages=stages, tail_brute=int(tail == "brute"))
        out3, _, _ = fresh.render(cam, Backend.params(w, h, spp, 50, seed=11, variant="mega"))
        assert np.array_equal(ref, out3), (stages, tail)
    fresh.close()


@pytest.mark.gpu
@pytest.mark.parametrize("n,kind", [(1, "one"), (2047, "uniform"), (2048, "few"), (2049, "sorted"), (70001, "uniform"), (1 << 20, "hot"),
                                    (3_000_017, "uniform"), (3_000_017, "few")])
def test_key_sort_groups_every_entry_by_key(be, n, kind):
    """rz_sort.cu directly (test hook): the entries come out grouped by ascending (key >> 4) — origin cell + octant; the low 4
    bits, the reach class, are ordered per work unit by the consumer — the indices (low 28 bits of the output word) are a
    permutation of the entries, the word's top four bits repeat the entry's reach class, and each index names an entry with the
    key stored beside it.  Order inside a group is free (the consumer does not depend on it)."""
    rng = np.random.default_rng(n)
    if kind == "uniform":
        keys = rng.integers(0, 65536, n, dtype=np.uint16)
    elif kind == "few":
        keys = rng.choice(np.array([0, 1, 15, 16, 255, 256, 40000, 65535], dtype=np.uint16), n)
    elif kind == "hot":     # one group holds 60 % of the entries: the shared-memory histogram's worst case
        keys = np.where(rng.random(n) < 0.6, np.uint16(12345), rng.integers(0, 65536, n, dtype=np.uint16)).astype(np.uint16)
    elif kind == "sorted":
        keys = np.sort(rng.integers(0, 3000, n, dtype=np.uint16))
    else:
        keys = np.array([777], dtype=np.uint16)
    ko, word = be.debug_sort_keys(keys)
    io = word & 0x0FFFFFFF
    assert np.array_equal(ko >> 4, np.sort(keys >> 4))
    assert np.array_equal(np.sort(io), np.arange(n, dtype=np.uint32))
    assert np.array_equal(keys[io], ko)
    assert np.array_equal(word >> 28, ko & 15)


@pytest.mark.gpu
def test_staged_render_with_big_sorted_passes_equals_single_kernel(scene42):
    """6.5 M paths in one pass: the sort runs over millions of entries per stage; the image must equal the one-kernel form."""
    w, spp = 1200, 8
    cam, h = cam_for(w)
    fresh = Backend((0,))
    fresh.upload_scene(scene42)
    img, _, _ = fresh.render(cam, Backend.params(w, h, spp, 50, seed=9, variant="mega"))
    again, _, _ = fresh.render(cam, Backend.params(w, h, spp, 50, seed=9, variant="mega"))
    single, _, _ = fresh.render(cam, Backend.params(w, h, spp, 50, seed=9, variant="mega_single"))
    assert fresh.timing()["variant"] == 4
    assert np.array_equal(img, again) and np.array_equal(img, single)
    fresh.close()


@pytest.mark.gpu
@pytest.mark.parametrize("seed", [1, 2, 3])
def test_staged_cull_is_conservative_on_hostile_scenes(seed):
    """Fast movers, a wide lens, the camera inside a sphere, spheres behind the camera, glass: the culled searches must
    find exactly the hits of the single brute-force kernel (and of the BVH kernel, up to its documented FP32 edge)."""
    rng = np.random.default_rng(seed)
    pool = rayz_b200.MemPool()
    ground = pool.add_diffuse(pool.add_checker(0.5, pool.add_solid((0.2, 0.3, 0.1)), pool.add_solid((0.9, 0.9, 0.9))))
    pool.add_sphere((0, -500, 0), 500.0, ground, (0, 0, 0))
    mats = [pool.add_diffuse(pool.add_solid(tuple(rng.uniform(0.2, 0.9, 3)))), pool.add_metallic(pool.add_solid((0.8, 0.8, 0.7)), 0.1),
            pool.add_dielectric(1.5)]
    for i in range(150):
        c = rng.uniform(-6, 6, 3); c[1] = abs(c[1]) * 0.5 + 0.3
        v = rng.uniform(-3, 3, 3) if i % 3 == 0 else (0, 0, 0)          # some travel several diameters per shutter interval
        pool.add_sphere(c, float(rng.uniform(0.15, 0.6)), mats[i % 3], v)
    pool.add_sphere((0, 1.0, 8.0), 1.5, mats[2], (0, 0, 0))            # the camera sits inside this glass sphere
    scene = pool.arrays()
    w, h, spp = 160, 90, 16
    cam = rayz_b200.Camera.init(50.0, 6.0, 8.0, (0, 1.0, 8.0), (0, 0.5, 0), (0, 1, 0), h, w).rz   # defocus angle 8 degrees
    be = Backend((0,))
    be.upload_scene(scene)
    ref, _, _ = be.render(cam, Backend.params(w, h, spp, 50, seed=seed, variant="mega_single"))
    be.set_tuning(tail_brute=1)                        # culled lists + brute-force tail: the same FP32 test on fewer spheres
    out, _, _ = be.render(cam, Backend.params(w, h, spp, 50, seed=seed, variant="mega"))
    assert np.array_equal(ref, out)
    for sectors in (0, 1, 2):                          # every direction field of the sort key (the default picks by the box's shape)
        be.set_tuning(key_sectors=sectors, second_stages=8)
        out, _, _ = be.render(cam, Backend.params(w, h, spp, 50, seed=seed, variant="mega"))
        assert np.array_equal(ref, out), sectors
    be.set_tuning(key_sectors=-1, second_stages=-1)
    be.set_tuning(tail_brute=0)                        # default: the tail of the paths walks the BVH (see below)
    out, _, _ = be.render(cam, Backend.params(w, h, spp, 50, seed=seed, variant="mega"))
    assert int((ref != out).any(axis=-1).sum()) <= 3 and float(np.abs(ref - out).mean()) < 1e-4
    # K3 prunes with (outward-rounded, exact) boxes while the brute-force kernels test every sphere with an FP32 test whose
    # apparent surface is fuzzy by ~3 |oc|^2 eps / (2 r): a grazing ray from far away can "hit" a sphere a hair outside its
    # box.  K3 then rejects what is in truth a miss, so it may differ from brute force in a pixel or two (measured: 0, 1, 0
    # of 14,400 on these scenes; padding the boxes by the fuzz bound makes them agree but costs K3 7-12 % and admits the
    # false hits).  Both stay far inside the tolerance against the f64 oracle.
    out, _, _ = be.render(cam, Backend.params(w, h, spp, 50, seed=seed, variant="bvh"))
    n_diff = int((ref != out).any(axis=-1).sum())
    assert n_diff <= 3, f"{n_diff} pixels differ between bvh and brute force"
    assert float(np.abs(ref - out).mean()) < 1e-4


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["all_moving", "all_static_cube", "one_static", "no_ground_flat"])
def test_staged_kernels_on_oddly_shaped_sphere_sets(kind):
    """The staged kernels keep stationary and moving spheres in separate parts of shared memory and of every list, and pick
    the sort key's direction field from the shape of the sphere box: sets with an empty part, a cubic box (octant keys) and a
    flat one (sector keys), with and without a huge sphere, must give the single brute-force kernel's image bit for bit."""
    rng = np.random.default_rng(11)
    pool = rayz_b200.MemPool()
    mats = [pool.add_diffuse(pool.add_solid((0.7, 0.4, 0.3))), pool.add_metallic(pool.add_solid((0.8, 0.8, 0.8)), 0.2), pool.add_dielectric(1.5)]
    n = 70
    for i in range(n):
        if kind == "all_static_cube":
            c, v = rng.uniform(-4, 4, 3), (0, 0, 0)
        elif kind == "all_moving":
            c, v = rng.uniform(-4, 4, 3) * (1, 0.2, 1), rng.uniform(-0.5, 0.5, 3)
        elif kind == "one_static":
            c, v = rng.uniform(-4, 4, 3) * (1, 0.2, 1), ((0, 0, 0) if i == 0 else rng.uniform(-0.5, 0.5, 3))
        else:
            c, v = rng.uniform(-5, 5, 3) * (1, 0.1, 1), ((0, 0, 0) if i % 2 else (0, 0.3, 0))
        pool.add_sphere(c, float(rng.uniform(0.2, 0.5)), mats[i % 3], v)
    if kind in ("all_static_cube", "one_static"):
        pool.add_sphere((0, -1005, 0), 1000.0, mats[0], (0, 0, 0) if kind == "all_static_cube" else (0, 0.1, 0))   # a huge sphere (a moving one too)
    w, h, spp = 192, 108, 8
    cam = rayz_b200.Camera.init(40.0, 10.0, 0.5, (9, 3, 7), (0, 0, 0), (0, 1, 0), h, w).rz
    be = Backend((0,))
    be.upload_scene(pool.arrays())
    ref, _, _ = be.render(cam, Backend.params(w, h, spp, 50, seed=4, variant="mega_single"))
    be.set_tuning(tail_brute=1)
    for sectors in (-1, 0, 1, 2):
        be.set_tuning(key_sectors=sectors)
        out, _, _ = be.render(cam, Backend.params(w, h, spp, 50, seed=4, variant="mega", collect_stats=True))
        assert be.timing()["sorted_stages"] >= 1 and be.stage_stats(1)["segments"] > 0      # the sorted-stage kernel really ran
        assert np.array_equal(ref, out), (kind, sectors)
    be.close()
    # which spheres stay outside the sphere box ("huge": culled by direction only) is a tuning matter, never an image matter:
    # the largest few (factor 1: everything above the median radius, capped at max(4, n / 32)), the default, none but the ground
    for factor in (1.0, 2.0, 1.0e6):
        be = Backend((0,))
        be.set_tuning(huge_factor=factor, tail_brute=1)    # (applies at the upload)
        be.upload_scene(pool.arrays())
        for sectors in (0, 1):
            be.set_tuning(key_sectors=sectors)
            out, _, _ = be.render(cam, Backend.params(w, h, spp, 50, seed=4, variant="mega", collect_stats=True))
            assert be.stage_stats(1)["segments"] > 0
            assert np.array_equal(ref, out), (kind, factor, sectors)
        be.close()


@pytest.mark.gpu
def test_reserve_then_render_and_auto_policy(scene42):
    """rayz_cuda_reserve pre-allocates the per-render buffers (before or after the scene upload) without changing results;
    RZ_VARIANT_AUTO resolves to the BVH kernel for small jobs and to the staged K1 for large ones (same image).  A staged
    BVH frame rendered as one shard of two, whose shard alone is below 2^26 paths: reserved by the frame's size too."""
    w, spp = 256, 8
    cam, h = cam_for(w)
    fresh = Backend((0,))
    p = Backend.params(w, h, spp, 50, seed=3, variant="mega")
    fresh.reserve(p)                                   # no scene yet
    fresh.upload_scene(scene42)
    fresh.reserve(p)                                   # idempotent
    a, _, _ = fresh.render(cam, p)
    b, _, _ = fresh.render(cam, Backend.params(w, h, spp, 50, seed=3, variant="auto"))
    assert fresh.timing()["variant"] == 3              # 256x144x8 paths: far below 2^26 -> BVH kernel
    assert np.array_equal(a, b)
    with pytest.raises(abi.BackendError):
        fresh.reserve(Backend.params(0, h, spp))
    w, spp = 1200, 100
    cam, h = cam_for(w)
    assert w * h * spp >= 1 << 26 > w * h * spp // 2
    p = Backend.params(w, h, spp, 50, seed=3, variant="bvh", shard_index=0, shard_count=2)
    fresh.reserve(p)
    c, c8, _ = fresh.render(cam, p)
    assert fresh.timing()["passes"] >= 1               # staged by the frame's size
    other = Backend((0,))
    other.upload_scene(scene42)
    d, d8, _ = other.render(cam, p)                    # no reserve
    assert np.array_equal(c, d) and np.array_equal(c8, d8)
    other.close()
    fresh.close()


@pytest.mark.gpu
def test_big_job_staged_bvh_equals_staged_bruteforce(scene42):
    """Above 2^26 paths per device the BVH variant also runs staged (coherent camera stage -> queue -> persistent kernel);
    81 M paths: it must equal the staged brute-force K1 and its own unstaged form bit for bit."""
    w, spp = 1200, 100
    cam, h = cam_for(w)
    be = Backend((0,))
    be.upload_scene(scene42)
    a, a8, _ = be.render(cam, Backend.params(w, h, spp, 50, seed=21, variant="mega"))
    assert be.timing()["passes"] >= 1
    b, b8, _ = be.render(cam, Backend.params(w, h, spp, 50, seed=21, variant="bvh", collect_stats=True))
    assert be.timing()["variant"] == 3 and be.timing()["passes"] >= 1
    st = be.stats()
    assert st["paths"] == w * h * spp and be.stage_stats(0)["segments"] == st["paths"]
    # brute-force stages against a BVH walk: equal up to the documented FP32-test-vs-exact-box edge (a pixel or two)
    assert int((a != b).any(axis=-1).sum()) <= 3 and float(np.abs(a - b).mean()) < 1e-5
    be.set_tuning(bvh_staged=0)
    c, _, _ = be.render(cam, Backend.params(w, h, spp, 50, seed=21, variant="bvh"))
    assert be.timing()["passes"] == 0
    assert np.array_equal(b, c)                       # the same tree walked staged or not: bit for bit
    be.set_tuning(bvh_staged=1, bvh_stages=2)
    d, _, _ = be.render(cam, Backend.params(w, h, spp, 50, seed=21, variant="bvh"))
    assert np.array_equal(b, d)
    be.close()


@pytest.mark.gpu
def test_staged_bvh_block_lists_on_odd_sizes_and_shards(scene42):
    """The staged K3's camera stage culls the tree once per 8 x 4-pixel block and searches the block's sphere list.  A frame
    whose width is no multiple of 8 and whose height is no multiple of 4 (partial blocks on two edges), full and in three
    shards of 3-row bands (blocks that straddle bands): the shards reproduce the full frame bit for bit, and the frame equals
    the unstaged kernel's per-ray walks up to the documented FP32-test-vs-exact-box edge."""
    w, spp = 1205, 84
    cam, h = cam_for(w)
    assert w % 8 and h % 4 and w * h * spp >= 1 << 26
    be = Backend((0,))
    be.upload_scene(scene42)
    full, full8, n = be.render(cam, Backend.params(w, h, spp, 50, seed=5, variant="bvh", collect_stats=True))
    assert n == w * h * spp and be.timing()["variant"] == 3 and be.timing()["passes"] >= 1
    st = be.stats()
    assert st["paths"] == n and st["ended_sky"] + st["ended_absorbed"] + st["ended_depth"] == n
    out, out8 = np.empty_like(full), np.empty_like(full8)
    for s in range(3):
        l, r, _ = be.render(cam, Backend.params(w, h, spp, 50, seed=5, variant="bvh", shard_index=s, shard_count=3, band_rows=3))
        assert be.timing()["passes"] >= 1                      # staged by the frame's size, not the shard's
        rows = [j for j in range(h) if (j // 3) % 3 == s]
        out[rows] = l; out8[rows] = r
    assert np.array_equal(out, full) and np.array_equal(out8, full8)
    be.set_tuning(bvh_staged=0)
    walk, _, _ = be.render(cam, Backend.params(w, h, spp, 50, seed=5, variant="bvh"))
    assert be.timing()["passes"] == 0
    assert int((walk != full).any(axis=-1).sum()) <= 3 and float(np.abs(walk - full).mean()) < 1e-5
    be.close()


# ---------------------------------------------------------------------------------------------
# BASELINE config 4: 99,856 spheres (randomBouncing with the grid loops widened to [-158, 158)), device-built LBVH.
# This is the code hit.zig:130-161,181-216 and geom.zig:38-66 are stressed by: rays travel hundreds of units, where the
# textbook FP32 discriminant loses 5 % of r^2 — the backend's cancellation-free sphere test (rz_sphere_test) is what keeps
# the image unbiased there.
# ---------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def scene100k():
    arrays = rayz_b200.random_bouncing(960, seed=42, grid_lo=-158, grid_hi=158).pool.arrays()
    assert len(arrays["sphere_radius"]) == 99856
    return arrays


@pytest.mark.gpu
def test_config4_primary_ids_bit_exact_100k_spheres(scene100k, orc):
    """K0 through the reference-shaped BVH (hit.zig:130-161 restated on the host) on 99,856 spheres at 960x540: bit-exact
    against the committed golden (tests/golden/make_golden.py) and against the oracle run here."""
    w = 960
    cam, h = cam_for(w)
    be = Backend((0,))
    be.upload_scene(scene100k)
    ids = be.primary_ids(cam, w, h, use_bvh=True)
    gold = np.load(os.path.join(GOLDEN, f"ids_config4_{w}x{h}.npz"))["ids"].astype(np.int32)
    assert gold.shape == ids.shape and (gold >= 0).sum() > 400000
    assert np.array_equal(ids, gold), f"{(ids != gold).sum()} of {gold.size} ids differ from the golden fixture"
    ocam, oh = orc.default_camera(w)
    ref = orc.Scene.from_arrays(scene100k).primary_ids(ocam, w, oh, use_bvh=True)
    assert np.array_equal(ids, ref)
    # brute force over all 99,856 spheres at a quarter of the pixels (1.3e10 f64 sphere tests) equals the BVH walk
    wb, hb = 480, 270
    camb, _ = cam_for(wb)
    ocamb, _ = orc.default_camera(wb)
    assert np.array_equal(be.primary_ids(camb, wb, hb, use_bvh=False), orc.Scene.from_arrays(scene100k).primary_ids(ocamb, wb, hb, use_bvh=True))
    be.close()


@pytest.mark.gpu
def test_config4_image_parity_100k_spheres_device_lbvh(scene100k, orc):
    """variant=bvh on the device-built LBVH vs two independently seeded oracle renders at 640x360, 64 spp: same
    floor-relative bars as test_image_parity_default_scene, segments per path within 1 %."""
    w, spp = 640, 64
    cam, h = cam_for(w)
    be = Backend((0,))                                   # >= 8192 spheres: LBVH built on the device
    be.upload_scene(scene100k)
    assert be.timing()["bvh_build_us"] > 0
    lin, _, n = be.render(cam, Backend.params(w, h, spp, 50, seed=1, variant="bvh", collect_stats=True))
    assert be.timing()["variant"] == 3 and n == w * h * spp and np.isfinite(lin).all()
    gst = be.stats()
    a, b, ost = _oracle_pair(orc, scene100k, w, h, spp)
    floor, got = compare(b, a), compare(lin[..., :3], a)
    print("floor", floor, "\ngpu  ", got, "\n", gst, "\n", ost)
    assert got["psnr"] >= floor["psnr"] - 0.3
    assert max(got["mae"]) <= max(floor["mae"]) * 1.05
    assert got["block_mae"] <= floor["block_mae"] * 1.15 + 1e-4
    sigma = (0.027 * 2 / (spp * w * h)) ** 0.5 * 3.0
    assert max(abs(x) for x in got["mean_diff"]) <= max(5e-4, 4 * sigma)
    # Segments per path within 1 % — of the paths that are not trapped.  The reference's tmin = 1e-10 (renderer.zig:107) lets
    # ~0.15 % of this scene's paths re-hit the sphere they just left at t ~ 2e-10, end up inside it and bounce there until
    # depth 50 (oracle ended_depth 22,279 of 14.7 M; DESIGN.md "known deviation"); the backend excludes self-hits analytically
    # (ended_depth 995).  Those trapped paths carry 50 segments each — 2.2 % of all segments — and nothing else differs:
    trapped = lambda st: (st["segments"] - 50 * st["ended_depth"]) / st["paths"]
    gs, os_ = trapped(gst), trapped(ost)
    print("segments per untrapped path: gpu", gs, "oracle", os_, "| raw", gst["segments"] / n, ost["segments"] / n)
    assert abs(gs - os_) / os_ < 0.01, (gs, os_)
    assert abs(gst["ended_sky"] / n - ost["ended_sky"] / n) < 2e-3
    assert abs(gst["hits_metallic"] - ost["hits_metallic"]) / ost["hits_metallic"] < 0.01
    assert abs(gst["hits_dielectric"] - ost["hits_dielectric"]) / ost["hits_dielectric"] < 0.015
    # AUTO on this scene is the same kernel (the set does not fit shared memory), staged or not by job size
    lin2, _, _ = be.render(cam, Backend.params(w, h, spp, 50, seed=1, variant="auto"))
    assert be.timing()["variant"] == 3 and np.array_equal(lin, lin2)
    be.close()


# ---------------------------------------------------------------------------------------------
# Reference features no reference scene uses (SURVEY 8f #4): checker textures whose children are checkers
# (CheckerTexture.value recurses through handles, material.zig:32-38) and the hollow-glass penultimateScene (rayz.zig:170-239).
# ---------------------------------------------------------------------------------------------
def _penultimate_pool(nested_checker: bool):
    """rayz_b200.penultimate_scene (rayz.zig:170-239); `nested_checker` swaps the ground's solid colour for a three-level
    checker: checker of (checker of solids, checker of (solid, checker of solids))."""
    pool = rayz_b200.penultimate_scene(256).pool
    if nested_checker:
        c1 = pool.add_checker(0.25, pool.add_solid((0.9, 0.1, 0.1)), pool.add_solid((0.1, 0.1, 0.9)))
        c2 = pool.add_checker(0.1, pool.add_solid((0.1, 0.8, 0.1)), pool.add_solid((0.9, 0.9, 0.1)))
        c3 = pool.add_checker(0.5, pool.add_solid((0.95, 0.95, 0.95)), c2)
        pool.mat_texture[pool.sphere_material[1]] = pool.add_checker(1.0, c1, c3)
    return pool


@pytest.mark.gpu
@pytest.mark.parametrize("nested", [False, True])
def test_penultimate_scene_and_nested_checkers(orc, nested):
    pool = _penultimate_pool(nested)
    arrays = pool.arrays()
    w, h, spp = 256, 144, 128
    args = (20.0, 3.4, 10.0, (-2, 2, 1), (0, 0, -1), (0, 1, 0), h, w)     # rayz.zig:170-180's camera
    cam, ocam = rayz_b200.Camera.init(*args).rz, orc.camera(*args)
    osc = orc.Scene.from_arrays(arrays)
    if nested:   # the texture walk itself, point by point, against the oracle's recursion (material.zig:32-38)
        root = int(arrays["mat_texture"][arrays["sphere_material"][1]])
        seen = {tuple(osc.texture_value(root, p)) for p in np.random.default_rng(1).uniform(-3, 3, (400, 3))}
        assert len(seen) == 5                                           # every leaf colour is reached (red, blue, white, green, yellow)
    be = Backend((0,))
    be.upload_scene(arrays)
    assert np.array_equal(be.primary_ids(cam, w, h), osc.primary_ids(ocam, w, h))
    a, _ = osc.render(ocam, w, h, spp, 50, seed=1, threads=0)
    b, _ = osc.render(ocam, w, h, spp, 50, seed=2, threads=0)
    floor = compare(b, a)
    for variant in ("mega_single", "bvh"):
        lin, _, _ = be.render(cam, Backend.params(w, h, spp, 50, seed=9, variant=variant))
        got = compare(lin[..., :3], a)
        print(variant, "floor", floor, "\ngpu  ", got)
        assert got["psnr"] >= floor["psnr"] - 0.3 and got["block_mae"] <= floor["block_mae"] * 1.2 + 1e-4
        assert max(abs(x) for x in got["mean_diff"]) <= 1.5e-3
    be.close()


# ---------------------------------------------------------------------------------------------
# Hardening: nothing is dropped silently, scratch reuse, shard invariance of AUTO.
# ---------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_capacity_overflow_is_an_error_not_a_darker_image(scene42):
    """A queue slot or traversal-stack entry that does not exist makes the render FAIL (RZ_ERR_INTERNAL) instead of
    dropping paths; the debug_* tuning fields shrink the capacities the kernels believe in."""
    w, spp = 320, 16
    cam, h = cam_for(w)
    be = Backend((0,))
    be.upload_scene(scene42)
    ok, _, _ = be.render(cam, Backend.params(w, h, spp, 50, seed=5, variant="mega"))
    be.set_tuning(debug_queue_cap=1000)
    with pytest.raises(abi.BackendError) as e:
        be.render(cam, Backend.params(w, h, spp, 50, seed=5, variant="mega"))
    assert e.value.code == -7 and "queue overflow" in str(e.value)
    be.set_tuning(debug_queue_cap=0, debug_stack_cap=2)
    with pytest.raises(abi.BackendError) as e:
        be.render(cam, Backend.params(w, h, spp, 50, seed=5, variant="bvh"))
    assert e.value.code == -7 and "stack overflow" in str(e.value)
    be.set_tuning(debug_stack_cap=0)
    again, _, _ = be.render(cam, Backend.params(w, h, spp, 50, seed=5, variant="mega"))
    assert np.array_equal(ok, again)                     # and the context is still good afterwards
    with pytest.raises(abi.BackendError):
        be.set_tuning(unit_entries=100)                  # not a multiple of 64
    with pytest.raises(abi.BackendError):
        be.set_tuning(queue_log2=40)
    be.close()


@pytest.mark.gpu
def test_wavefront_scratch_reuse_large_then_small(scene42):
    """The wavefront's slot pool is reused across renders: a job that fills the pool followed by a smaller one on the same
    context must rebuild the whole free list (round-1 bug: stale top of the stack handed out slots twice)."""
    be = Backend((0,))
    be.upload_scene(scene42)
    cam_big, hb = cam_for(640)
    big, _, _ = be.render(cam_big, Backend.params(640, hb, 24, 50, seed=3, variant="wavefront"))      # 5.5 M paths > 2^21 slots
    ref_big, _, _ = be.render(cam_big, Backend.params(640, hb, 24, 50, seed=3, variant="mega_single"))
    assert np.array_equal(big, ref_big)
    for w, spp in ((400, 16), (320, 12), (64, 4)):       # 1.4 M (between 2^20 and 2^21), 0.7 M, tiny
        cam, h = cam_for(w)
        small, _, _ = be.render(cam, Backend.params(w, h, spp, 50, seed=4, variant="wavefront"))
        ref, _, _ = be.render(cam, Backend.params(w, h, spp, 50, seed=4, variant="mega_single"))
        assert np.array_equal(small, ref), (w, spp)
    be.close()


@pytest.mark.gpu
def test_auto_variant_does_not_depend_on_the_sharding(scene42):
    """include/rayz_cuda.h promises that any sharding reproduces the full-frame render bit for bit.  AUTO therefore picks
    its kernels from the whole frame's size, never from a shard's share: 1200x675 at 100 spp is an 81 M-path frame (staged
    K1); each of 8 shards holds 10 M paths and must still run the staged K1, with the same number of sorted stages."""
    w, spp = 1200, 100
    cam, h = cam_for(w)
    be = Backend((0,))
    be.upload_scene(scene42)
    full, full8, _ = be.render(cam, Backend.params(w, h, spp, 50, seed=13, variant="auto"))
    assert be.timing()["variant"] == 1
    out, out8 = np.empty_like(full), np.empty_like(full8)
    for s in range(8):
        l, r, _ = be.render(cam, Backend.params(w, h, spp, 50, seed=13, variant="auto", shard_index=s, shard_count=8, band_rows=4))
        assert be.timing()["variant"] == 1
        rows = [j for j in range(h) if (j // 4) % 8 == s]
        out[rows] = l; out8[rows] = r
    assert np.array_equal(out, full) and np.array_equal(out8, full8)
    small_be = Backend((0,))
    small_be.set_tuning(queue_log2=20)                   # a device short of memory steps the pass size down: same image
    small_be.upload_scene(scene42)
    small, _, _ = small_be.render(cam, Backend.params(w, h, spp, 50, seed=13, variant="auto"))
    assert small_be.timing()["passes"] > 8 and np.array_equal(small, full)
    be.close(); small_be.close()
