"""GPU tests of the pixel filters (include/rayz_cuda.h "RZ_RENDER_FILTER").

Each camera sample of a filtered render starts at px + w(u), w the filter's warp; nothing else about a path changes.  So:
  * every kernel family's camera rays are checked against the f64 restatement of the same samples (filter_replay): at depth 1
    a pixel of a 1-spp frame is lit exactly when its camera ray misses, and the mattes' first-hit ids equal the replay's;
  * the kernels that share a family agree bit for bit on frames of >= 2^26 paths (the staged forms and their widened culls),
    and batches, shards, devices and adaptive counts keep their bit-for-bit guarantees;
  * the filter's shape shows through the public interface: the mattes' coverage of a sphere's silhouette pixels is the f64
    quadrature of the filter, and not the box's;
  * guides and the denoiser follow the frame's filter, refusals touch nothing, and the C++ host's --filter matches Backend."""
import ctypes as C
import io
import os
import subprocess

import numpy as np
import pytest

import rayz_b200
from rayz_b200 import Backend
from rayz_b200 import _abi as abi
import filter_replay as fr
import replay_scenes

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SEED = 11
FILTERS = [("tent", None), ("gaussian", None), ("blackman-harris", None)]
VARIANTS = [("auto", {}), ("mega", {"tail_brute": 0}), ("mega", {"tail_brute": 1}), ("mega_single", {}), ("wavefront", {}),
            ("bvh", {})]
SAMPLERS = {"philox": {}, "sobol": {"sobol": True}}


def cam_for(w, defocus=0.6):
    h = int(w / rayz_b200.ASPECT_RATIO)
    return rayz_b200.Camera.init(20.0, 10.0, defocus, (13, 2, 3), (0, 0, 0), (0, 1, 0), h, w).rz, h


@pytest.fixture(scope="module")
def bench_scene():
    return rayz_b200.random_bouncing(1200, seed=42).pool.arrays()


@pytest.fixture(scope="module")
def be():
    b = Backend((0,))
    yield b
    b.close()


# ------------------------------------------------------------------------------- 1. every family's rays against the f64 replay
def _replay_cases():
    arrays1, cam1 = replay_scenes.config1(64, 36)
    am, cams, w, h = replay_scenes.all_materials()
    return {"config1": (arrays1, cam1, 64, 36), "allmat": (am, cams["outside"], w, h)}


@pytest.mark.parametrize("sampler", list(SAMPLERS))
@pytest.mark.parametrize("pixel_filter,filter_width", FILTERS)
@pytest.mark.parametrize("scene", ["config1", "allmat"])
def test_every_family_traces_the_replayed_camera_rays(be, scene, pixel_filter, filter_width, sampler):
    """1 spp, depth 1: a path adds the sky's radiance when its camera ray misses and nothing when it hits, so every kernel
    family's frame says which filtered camera rays hit.  Against the f64 replay of the same samples, every robust ray (not
    within 1e-4 of a silhouette or of a second root) agrees, with zero exceptions; the mattes' first-hit ids equal the
    replay's ids on robust rays, and the fragile fraction stays below 2 %."""
    arrays, cam, w, h = _replay_cases()[scene]
    be.upload_scene(arrays)
    o, d, t = fr.camera_rays(cam, w, h, 0, 1, SEED, sampler, pixel_filter, filter_width)
    ids, robust = fr.first_hits_robust(arrays, o, d, t)
    ids, robust = ids[..., 0], robust[..., 0]
    frag = 1.0 - float(robust.mean())
    assert frag <= 0.02, f"fragile fraction {frag:.3%}"
    lit_sky = d[..., 0, 1] > -0.99                 # the sky's radiance is 0 straight down
    miss = ids < 0
    if scene == "config1":   # the all-materials scene has no sky in view: there the mattes' ids carry the check
        assert miss.mean() > 0.1 and (~miss).mean() > 0.5
    try:
        for variant, tun in VARIANTS:
            be.set_tuning(**{"tail_brute": 0, **tun})
            for stats in (False, True):
                p = Backend.params(w, h, 1, 1, seed=SEED, variant=variant, collect_stats=stats, pixel_filter=pixel_filter,
                                   filter_width=filter_width, **SAMPLERS[sampler])
                lin, _, _ = be.render(cam, p, want_rgb8=False)
                lit = (lin[..., :3] > 0).any(axis=-1)
                bad = robust & lit_sky & (lit != miss)
                assert not bad.any(), f"{variant} {tun} stats {stats}: {int(bad.sum())} robust pixels disagree with the replay"
    finally:
        be.set_tuning(tail_brute=0)
    got, _ = be.mattes(cam, Backend.params(w, h, 1, 50, seed=SEED, variant="bvh", pixel_filter=pixel_filter,
                                           filter_width=filter_width, **SAMPLERS[sampler]), 1)
    bad = robust & (got[..., 0] != ids)
    assert not bad.any(), f"mattes: {int(bad.sum())} robust samples with another first hit than the replay"
    # and the filter is not the box: the box's rays disagree somewhere
    ob, db, tb = fr.camera_rays(cam, w, h, 0, 1, SEED, sampler)
    assert (np.abs(db - d) > 1e-4).any()


# ------------------------------------------------------------------------------- 2. bit for bit on >= 2^26 paths
BIG = [("gaussian", 4.0), ("blackman-harris", None)]


@pytest.mark.parametrize("pixel_filter,filter_width", BIG)
def test_families_shards_and_staging_agree_bitwise(bench_scene, pixel_filter, filter_width):
    """The benchmark scene (defocus, motion blur) at 1200 x 675 x 84 spp = 68 M paths, so that the staged K1 and the staged
    K3 run with their widened tile and block cones: staged MEGA == MEGA_SINGLE == WAVEFRONT, staged BVH == unstaged BVH, and
    shards reassemble the full frame."""
    w, spp = 1200, 84
    cam, h = cam_for(w)
    assert w * h * spp >= 1 << 26
    be = Backend((0,))
    be.upload_scene(bench_scene)
    kw = dict(seed=21, pixel_filter=pixel_filter, filter_width=filter_width)
    try:
        mega, mega8, n = be.render(cam, Backend.params(w, h, spp, 50, variant="mega", **kw))
        assert n == w * h * spp and be.timing()["passes"] >= 1
        for v in ("mega_single", "wavefront"):
            x, x8, _ = be.render(cam, Backend.params(w, h, spp, 50, variant=v, **kw))
            assert np.array_equal(x, mega) and np.array_equal(x8, mega8), v
        box, _, _ = be.render(cam, Backend.params(w, h, spp, 50, variant="mega", seed=21))
        assert not np.array_equal(box, mega)
        bvh, bvh8, _ = be.render(cam, Backend.params(w, h, spp, 50, variant="bvh", **kw))
        assert be.timing()["variant"] == 3 and be.timing()["passes"] >= 1
        be.set_tuning(bvh_staged=0)
        walk, _, _ = be.render(cam, Backend.params(w, h, spp, 50, variant="bvh", **kw))
        assert be.timing()["passes"] == 0
        assert np.array_equal(walk, bvh)
        be.set_tuning(bvh_staged=1)
        for variant, full, full8 in (("mega", mega, mega8), ("bvh", bvh, bvh8)):
            for count, band in ((2, 1), (3, 4)):
                out, out8 = np.empty_like(full), np.empty_like(full8)
                for s in range(count):
                    l, r, _ = be.render(cam, Backend.params(w, h, spp, 50, variant=variant, shard_index=s, shard_count=count,
                                                            band_rows=band, **kw))
                    rows = [j for j in range(h) if (j // band) % count == s]
                    out[rows] = l
                    out8[rows] = r
                assert np.array_equal(out, full) and np.array_equal(out8, full8), (variant, count, band)
    finally:
        be.close()


def _n_gpus():
    import torch
    return torch.cuda.device_count()


@pytest.mark.skipif("_n_gpus() < 2")
def test_multi_device_equals_single_device(bench_scene):
    w, spp = 1200, 84
    cam, h = cam_for(w)
    one, many = Backend((0,)), Backend(tuple(range(min(_n_gpus(), 4))))
    for b in (one, many):
        b.upload_scene(bench_scene)
    for pixel_filter, filter_width in BIG:
        for variant in ("mega", "bvh"):
            p = Backend.params(w, h, spp, 50, seed=4, variant=variant, pixel_filter=pixel_filter, filter_width=filter_width)
            a, a8, _ = one.render(cam, p)
            b, b8, _ = many.render(cam, p)
            assert np.array_equal(a, b) and np.array_equal(a8, b8), (pixel_filter, variant)
    one.close()
    many.close()


# ------------------------------------------------------------------------------- 3. batches
W = 160


@pytest.fixture(scope="module")
def small(be):
    be.upload_scene(rayz_b200.random_bouncing(W, seed=42).pool.arrays())
    return be


@pytest.mark.parametrize("variant", ["mega", "bvh", "wavefront"])
def test_batches_equal_one_render_and_another_filter_is_refused(small, variant):
    be = small
    cam, h = cam_for(W)
    kw = dict(seed=5, variant=variant, moments=True, pixel_filter="gaussian", filter_width=2.5, sobol=True)
    one, one8, _ = be.render(cam, Backend.params(W, h, 24, 50, **kw))
    err1, _ = be.noise()
    be.render(cam, Backend.params(W, h, 10, 50, **kw))
    for other in (dict(pixel_filter="gaussian", filter_width=2.0), dict(pixel_filter="tent", filter_width=2.5),
                  dict(pixel_filter="box", filter_width=None)):
        bad = Backend.params(W, h, 14, 50, sample_offset=10, accumulate=True, **{**kw, **other})
        lin = np.full((h, W, 4), 7.0, np.float32)
        rc = be.lib.rayz_cuda_render(be._h, C.byref(cam), C.byref(bad), lin.ctypes.data, None, None)
        assert rc == -1 and b"pixel filter" in be.lib.rayz_cuda_last_error(), be.lib.rayz_cuda_last_error()
        assert (lin == 7.0).all()
    two, two8, _ = be.render(cam, Backend.params(W, h, 14, 50, sample_offset=10, accumulate=True, **kw))
    err2, _ = be.noise()
    assert np.array_equal(two, one) and np.array_equal(two8, one8) and np.array_equal(err2, err1)


# ------------------------------------------------------------------------------- 4. adaptive and passes
@pytest.mark.parametrize("variant", ["bvh", "mega"])
def test_adaptive_pixels_equal_uniform_renders_of_their_count(small, variant):
    be = small
    cam, h = cam_for(W)
    kw = dict(seed=3, sample_offset=5, variant=variant, pixel_filter="blackman-harris", filter_width=3.0)
    be.render(cam, Backend.params(W, h, 4, 50, moments=True, **kw))
    target = float(np.quantile(be.noise(0.0)[0], 0.5) / 4)
    lin, rgb8, _, _ = be.render_to_noise(cam, Backend.params(W, h, 4, 50, **kw), target, 64, adaptive=True)
    err, _ = be.noise(target)
    counts = be.pixel_samples()
    assert len(np.unique(counts)) >= 3
    for c in np.unique(counts):
        m = counts == c
        u, u8, _ = be.render(cam, Backend.params(W, h, int(c), 50, moments=True, **kw))
        ue, _ = be.noise(0.0)
        for got, want, name in ((lin, u, "linear"), (rgb8, u8, "rgb8"), (err, ue, "err")):
            assert np.array_equal(got[m], want[m]), f"{variant}, count {c}: {name}"


def test_passes_sum_to_the_filtered_frame(small):
    be = small
    cam, h = cam_for(W)
    for variant in ("mega", "bvh"):
        lin, _, _ = be.render(cam, Backend.params(W, h, 16, 50, seed=2, variant=variant, passes=True, pixel_filter="tent",
                                                  filter_width=4.0))
        planes = be.passes()
        total = planes[..., :3].astype(np.float64).sum(axis=0)
        assert np.allclose(total, lin[..., :3], rtol=1e-5, atol=1e-6), variant
        plain, _, _ = be.render(cam, Backend.params(W, h, 16, 50, seed=2, variant=variant, pixel_filter="tent", filter_width=4.0))
        assert np.array_equal(plain, lin)


# ------------------------------------------------------------------------------- 5. the filter's shape, seen through the mattes
def _one_sphere():
    pool = rayz_b200.MemPool()
    pool.add_sphere((0.0, 0.0, 0.0), 0.6, pool.add_diffuse(pool.add_solid((0.5, 0.5, 0.5))))
    w, h, s = 64, 48, 0.004
    cam = abi.RzCamera()
    cam.look_from[:] = (0.0, 0.0, 10.0)
    cam.px_du[:] = (s, 0.0, 0.0)
    cam.px_dv[:] = (0.0, -s, 0.0)
    cam.px_origin[:] = (-(w - 1) / 2 * s + 0.0013, (h - 1) / 2 * s - 0.0007, 9.0)   # off the pixel grid's symmetry
    return pool.arrays(), cam, w, h


def _expected_coverage(cam, w, h, kind, width, n=128):
    """f64 quadrature of the filter over each pixel: the mean over an n x n midpoint grid of jitter uniforms of whether the
    pinhole ray through px + w(u) hits the sphere (centre 0, radius 0.6)."""
    um = (np.arange(n) + 0.5) / n
    off = um - 0.5 if kind == fr.BOX else fr.filter_warp(kind, width, um)
    o = np.array(cam.look_from[:])
    du, dv, p0 = np.array(cam.px_du[:]), np.array(cam.px_dv[:]), np.array(cam.px_origin[:])
    cov = np.zeros((h, w))
    for j in range(h):
        x = np.arange(w)[:, None, None] + off[None, :, None]          # [w, n, 1]
        y = j + off[None, None, :]                                      # [1, 1, n]
        d = du * x[..., None] + dv * y[..., None] + (p0 - o)           # [w, n, n, 3]
        d = d / np.linalg.norm(d, axis=-1, keepdims=True)
        oc = -o
        b = d @ oc
        l2 = oc @ oc - b * b
        cov[j] = ((l2 < 0.36) & (b > 0)).mean(axis=(1, 2))
    return cov


@pytest.mark.parametrize("pixel_filter,filter_width", [("gaussian", 4.0), ("tent", 2.0), ("blackman-harris", 4.0)])
def test_coverage_of_a_silhouette_is_the_filters(be, pixel_filter, filter_width):
    arrays, cam, w, h = _one_sphere()
    be.upload_scene(arrays)
    spp = 1024
    kind = fr.KINDS[pixel_filter]
    ids, cov = be.mattes(cam, Backend.params(w, h, spp, 50, seed=9, variant="bvh", pixel_filter=pixel_filter,
                                             filter_width=filter_width), 2)
    got = np.where(ids == 0, cov, 0.0).sum(axis=-1).astype(np.float64)
    want = _expected_coverage(cam, w, h, kind, filter_width)
    box = _expected_coverage(cam, w, h, fr.BOX, 1.0)
    edge = (want > 0.05) & (want < 0.95)
    assert edge.sum() > 100

    def within(p):
        return np.abs(got - p) <= 4.0 * np.sqrt(np.maximum(p * (1 - p), 1e-12) / spp) + 2.0 / spp

    ok, box_ok = within(want)[edge], within(box)[edge]
    print(f"{pixel_filter} {filter_width} px: {int(edge.sum())} silhouette pixels, all within the filter's bound: {ok.all()}; "
          f"the box's coverage fails on {1 - box_ok.mean():.1%} of them")
    assert ok.all(), f"{int((~ok).sum())} pixels off the filter's coverage"
    assert box_ok.mean() < 0.5, "the box's coverage would pass on most silhouette pixels: the check does not tell the filters apart"


# ------------------------------------------------------------------------------- 6. guides and the denoiser
@pytest.mark.parametrize("sampler", list(SAMPLERS))
def test_guides_follow_the_frames_rays(small, sampler):
    be = small
    cam, h = cam_for(W)
    kw = dict(seed=8, pixel_filter="gaussian", filter_width=3.5, **SAMPLERS[sampler])
    alb, _ = be.guides(cam, Backend.params(W, h, 1, 50, variant="bvh", **kw))
    for variant in ("bvh", "mega"):
        lin, _, _ = be.render(cam, Backend.params(W, h, 1, 1, variant=variant, **kw))
        sky = (lin[..., :3] > 0).any(axis=-1)
        assert np.array_equal(alb[..., 3] == 0, sky), variant
    box, _ = be.guides(cam, Backend.params(W, h, 1, 50, variant="bvh", seed=8, **SAMPLERS[sampler]))
    assert not np.array_equal(box, alb)


def test_denoise_takes_guides_of_the_frames_filter_only(small):
    be = small
    cam, h = cam_for(W)
    kw = dict(seed=6, variant="bvh", pixel_filter="tent", filter_width=3.0)
    be.render(cam, Backend.params(W, h, 8, 50, moments=True, **kw))
    be.guides(cam, Backend.params(W, h, 8, 50, **kw))
    lin, rgb8 = be.denoise()
    assert np.isfinite(lin).all()
    for other in (dict(pixel_filter="tent", filter_width=2.0), dict(pixel_filter="gaussian", filter_width=3.0), {}):
        be.guides(cam, Backend.params(W, h, 8, 50, **{**kw, **other}) if other else Backend.params(W, h, 8, 50, seed=6, variant="bvh"))
        rc = be.lib.rayz_cuda_denoise(be._h, None, None, None)
        assert rc == -1 and b"pixel filter" in be.lib.rayz_cuda_last_error(), be.lib.rayz_cuda_last_error()
    be.guides(cam, Backend.params(W, h, 8, 50, **kw))
    again = be.denoise()
    assert np.array_equal(again[0], lin) and np.array_equal(again[1], rgb8)


# ------------------------------------------------------------------------------- 7. refusals
def test_refusals_touch_nothing(small):
    be = small
    cam, h = cam_for(W)
    lib = be.lib
    base = Backend.params(W, h, 4, 50, seed=1, variant="bvh", moments=True)
    want, want8, _ = be.render(cam, base)
    err0, _ = be.noise()
    bad_fields = [abi.render_filter(abi.FILTER_TENT, 1), abi.render_filter(abi.FILTER_GAUSSIAN, 15),
                  abi.render_filter(abi.FILTER_BLACKMAN_HARRIS, 65), abi.render_filter(abi.FILTER_TENT, 255),
                  abi.render_filter(abi.FILTER_BOX, 16), abi.render_filter(abi.FILTER_BOX, 32)]
    lin = np.full((h, W, 4), 7.0, np.float32)
    a4 = np.full((h, W, 4), 7.0, np.float32)
    ids = np.full((h, W, 2), 77, np.int32)
    cv = np.full((h, W, 2), 0.5, np.float32)
    n, nz = C.c_uint64(), abi.RzNoise()
    for field in bad_fields:
        p = abi.RzRenderParams.from_buffer_copy(base)
        p.flags |= field
        q = abi.RzRenderParams.from_buffer_copy(p)
        q.flags |= abi.RENDER_ACCUMULATE
        q.sample_offset = 4
        g = abi.RzRenderParams.from_buffer_copy(p)
        g.flags &= ~abi.RENDER_MOMENTS
        calls = {
            "render": lambda: lib.rayz_cuda_render(be._h, C.byref(cam), C.byref(p), lin.ctypes.data, None, None),
            "accumulate": lambda: lib.rayz_cuda_render(be._h, C.byref(cam), C.byref(q), lin.ctypes.data, None, None),
            "reserve": lambda: lib.rayz_cuda_reserve(be._h, C.byref(p)),
            "to_noise": lambda: lib.rayz_cuda_render_to_noise(be._h, C.byref(cam), C.byref(p), 0.01, 16, lin.ctypes.data, None,
                                                              C.byref(n), C.byref(nz)),
            "guides": lambda: lib.rayz_cuda_render_guides(be._h, C.byref(cam), C.byref(g), a4.ctypes.data, None),
            "mattes": lambda: lib.rayz_cuda_render_mattes(be._h, C.byref(cam), C.byref(g), 2, ids.ctypes.data, cv.ctypes.data),
        }
        for name, call in calls.items():
            rc = call()
            msg = lib.rayz_cuda_last_error()
            assert rc == -1 and (b"width" in msg), (hex(field), name, rc, msg)
    assert (lin == 7.0).all() and (a4 == 7.0).all() and (ids == 77).all() and (cv == 0.5).all()
    err, _ = be.noise()
    assert np.array_equal(err, err0)
    nxt, nxt8, _ = be.render(cam, Backend.params(W, h, 4, 50, seed=1, variant="bvh", moments=True, sample_offset=4, accumulate=True))
    full, full8, _ = be.render(cam, Backend.params(W, h, 8, 50, seed=1, variant="bvh", moments=True))
    assert np.array_equal(nxt, full) and np.array_equal(nxt8, full8)


# ------------------------------------------------------------------------------- 8. the C++ host
def test_cpp_host_filter_matches_backend(tmp_path):
    subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "host")], check=True)
    exe = os.path.join(ROOT, "host", "_build", "rayz_host")
    out = tmp_path / "o.ppm"
    r = subprocess.run([exe, str(W), str(out), "--spp", "8", "--seed", "42", "--render-seed", "5", "--filter", "gaussian:3"],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    t = rayz_b200.random_bouncing(W, seed=42)
    t.samples_per_px, t.seed, t.pixel_filter, t.filter_width = 8, 5, "gaussian", 3.0
    t.render()
    f = io.StringIO()
    t.img.writePPM(f)
    assert out.read_bytes() == f.getvalue().encode()
    t.pixel_filter = "box"
    t.filter_width = None
    t.render()
    g = io.StringIO()
    t.img.writePPM(g)
    assert out.read_bytes() != g.getvalue().encode()
    t.backend.close()
    for bad in ("mitchell", "gaussian:0.5", "tent:1.03"):
        r = subprocess.run([exe, "16", str(tmp_path / "x.ppm"), "--filter", bad], capture_output=True, text=True, timeout=300)
        assert r.returncode != 0, bad
