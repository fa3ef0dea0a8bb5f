"""GPU tests of progressive rendering: RZ_RENDER_ACCUMULATE batches, the RZ_RENDER_MOMENTS noise estimate
(rayz_cuda_noise) and rayz_cuda_render_to_noise.

Radiance and the luminance second moment are summed in 64-bit fixed point, so batches [0,a) + [a,b) + ... of one kernel
family must reproduce a single render of all the samples bit for bit: image and error buffer alike."""
import numpy as np
import pytest

import oracle
import rayz_b200
from rayz_b200 import Backend
from rayz_b200 import _abi as abi

pytestmark = pytest.mark.gpu
LUMA = np.array([0.2126, 0.7152, 0.0722])
FLOOR = 1e-4   # RZ_NOISE_Y_FLOOR


@pytest.fixture(scope="module")
def scene():
    return rayz_b200.random_bouncing(160, seed=42).pool.arrays()


@pytest.fixture(scope="module")
def be(scene):
    b = Backend((0,))
    b.upload_scene(scene)
    yield b
    b.close()


def cam_for(w):
    h = int(w / rayz_b200.ASPECT_RATIO)
    return rayz_b200.Camera.init(20.0, 10.0, 0.6, (13, 2, 3), (0, 0, 0), (0, 1, 0), h, w).rz, h


def batches(be, cam, w, h, cuts, variant, seed=3, **kw):
    """Renders the sample ranges [cuts[k], cuts[k+1]) as RZ_RENDER_ACCUMULATE batches -> (linear, rgb8, err, summary)."""
    for k in range(len(cuts) - 1):
        p = Backend.params(w, h, cuts[k + 1] - cuts[k], 50, seed=seed, sample_offset=cuts[k], variant=variant, moments=True,
                           accumulate=k > 0, **kw)
        lin, rgb8, n = be.render(cam, p)
        assert n == be.shard_rows(p) * w * (cuts[k + 1] - cuts[k])   # the paths of this call only
    err, nz = be.noise(2 / 255)
    return lin, rgb8, err, nz


def single(be, cam, w, h, spp, variant, seed=3, moments=True, **kw):
    lin, rgb8, _ = be.render(cam, Backend.params(w, h, spp, 50, seed=seed, variant=variant, moments=moments, **kw))
    if not moments:
        return lin, rgb8, None, None
    err, nz = be.noise(2 / 255)
    return lin, rgb8, err, nz


def assert_same(a, b):
    for x, y, name in zip(a[:3], b[:3], ("linear", "rgb8", "err")):
        assert x.shape == y.shape and np.array_equal(x, y), f"{name}: {int((x != y).sum())} values differ"


# ------------------------------------------------------------------------------- 1. batches == one render, bit for bit
@pytest.mark.parametrize("variant", ["mega", "mega_single", "wavefront", "bvh"])
def test_batches_equal_single_render_bitwise(be, variant):
    w = 160
    cam, h = cam_for(w)
    one = single(be, cam, w, h, 24, variant)
    acc = batches(be, cam, w, h, [0, 3, 8, 24], variant)
    assert_same(acc, one)
    assert acc[3] == one[3] and acc[3]["samples"] == 24 and acc[3]["n_pixels"] == w * h
    assert np.isfinite(one[2]).all() and (one[2] >= 0).all() and one[3]["rms_err"] > 0
    # three shards of 3-row bands: every shard accumulates its own rows, and the shards assemble the full frame
    full = [np.empty_like(x) for x in one[:3]]
    for s in range(3):
        kw = dict(shard_index=s, shard_count=3, band_rows=3)
        o = single(be, cam, w, h, 24, variant, **kw)
        a = batches(be, cam, w, h, [0, 3, 8, 24], variant, **kw)
        assert_same(a, o)
        rows = [j for j in range(h) if (j // 3) % 3 == s]
        for f, x in zip(full, a[:3]):
            f[rows] = x
    for f, x in zip(full, one[:3]):
        assert np.array_equal(f, x)


# ------------------------------------------------------------------------------- 2. moments change no pixel
@pytest.mark.parametrize("variant", ["mega", "mega_single", "wavefront", "bvh"])
def test_moments_change_no_pixel(be, variant):
    w = 160
    cam, h = cam_for(w)
    off = single(be, cam, w, h, 16, variant, seed=8, moments=False)
    on = single(be, cam, w, h, 16, variant, seed=8, moments=True)
    assert np.array_equal(off[0], on[0]) and np.array_equal(off[1], on[1])


# ------------------------------------------------------------------------------- 3. refusals
def _code(fn):
    with pytest.raises(abi.BackendError) as e:
        fn()
    return e.value.code


def test_accumulate_refusals_leave_the_sums_intact(be, scene):
    w, v = 160, "mega"
    cam, h = cam_for(w)
    want = single(be, cam, w, h, 12, v, seed=21)
    P = lambda **kw: Backend.params(**({"width": w, "height": h, "spp": 8, "max_depth": 50, "seed": 21, "sample_offset": 4,
                                        "variant": v, "moments": True, "accumulate": True} | kw))
    be.render(cam, Backend.params(w, h, 4, 50, seed=21, variant=v, moments=True))   # batch [0, 4)
    cam2, _ = cam_for(w)
    cam2.look_from[0] += 1e-9
    cam3, h3 = cam_for(192)
    refused = {
        "width": (cam3, P(width=192, height=h3)), "height": (cam, P(height=h - 1)), "shard": (cam, P(shard_index=0, shard_count=2)),
        "band_rows": (cam, P(shard_index=0, shard_count=1, band_rows=8)), "seed": (cam, P(seed=22)), "max_depth": (cam, P(max_depth=49)),
        "t_min": (cam, P(t_min=1e-3)), "camera": (cam2, P()), "moments": (cam, P(moments=False)), "offset_gap": (cam, P(sample_offset=5)),
        "offset_overlap": (cam, P(sample_offset=0)), "count": (cam, P(spp=0xFFFFFFFF - 3)),
    }
    for name, (c, p) in refused.items():
        assert _code(lambda: be.render(c, p)) == -1, name
        assert b"RZ_RENDER_ACCUMULATE refused" in be.lib.rayz_cuda_last_error(), name
    lin, rgb8, _ = be.render(cam, P())   # the valid batch [4, 12) after all of them
    err, nz = be.noise(2 / 255)
    assert_same((lin, rgb8, err), want)
    assert nz == want[3]

    # a scene upload, or a reserve of another shape, ends the accumulation
    be.render(cam, Backend.params(w, h, 4, 50, seed=21, variant=v, moments=True))
    be.reserve(Backend.params(192, h3, 4, 50, variant="bvh"))
    assert _code(lambda: be.render(cam, P())) == -1
    be.render(cam, Backend.params(w, h, 4, 50, seed=21, variant=v, moments=True))
    be.reserve(Backend.params(w, h, 4, 50, variant="bvh"))   # the same shape: the sums stay
    be.render(cam, P())
    assert np.array_equal(be.noise(2 / 255)[0], want[2])
    be.upload_scene(scene)
    assert _code(lambda: be.render(cam, P(sample_offset=12))) == -1
    assert _code(lambda: be.noise(2 / 255)) == -1

    # a batch that fails (a queue capacity the kernels believe in is exceeded: RZ_ERR_INTERNAL) ends the accumulation
    be.render(cam, Backend.params(w, h, 4, 50, seed=21, variant=v, moments=True))
    be.set_tuning(debug_queue_cap=1000)
    try:
        assert _code(lambda: be.render(cam, P())) == -7
    finally:
        be.set_tuning(debug_queue_cap=0)
    assert _code(lambda: be.render(cam, P())) == -1
    assert _code(lambda: be.noise(2 / 255)) == -1

    # the same through rayz_cuda_render_device(sync = 0): the next batch reads the failed batch's error word first
    be.render(cam, Backend.params(w, h, 4, 50, seed=21, variant=v, moments=True))
    be.set_tuning(debug_queue_cap=1000)
    try:
        be.render_device(cam, P(), sync=False)
    finally:
        be.set_tuning(debug_queue_cap=0)
    assert _code(lambda: be.render(cam, P(sample_offset=12))) == -1
    # ... and an asynchronous batch that succeeded is added to as usual
    be.render_device(cam, Backend.params(w, h, 4, 50, seed=21, variant=v, moments=True), sync=False)
    lin, rgb8, _ = be.render(cam, P())
    err, _ = be.noise(2 / 255)
    assert_same((lin, rgb8, err), want)

    # noise needs the second moment
    be.render(cam, Backend.params(w, h, 4, 50, seed=21, variant=v))
    assert _code(lambda: be.noise(2 / 255)) == -1
    assert _code(lambda: Backend((0,)).noise(2 / 255)) == -1


# ------------------------------------------------------------------------------- 4. the estimator is right
def test_noise_estimate_matches_empirical_and_oracle_variance(be, scene):
    """32 seeds x 16 spp at 160x90: the estimated variance of the pixel mean (sigma^2 = s^2 / n, from the per-pixel second
    moment) against the variance of the mean luminance across the seeds; and the per-path variance s^2 against the oracle's."""
    w, spp, n_seeds = 160, 16, 32
    cam, h = cam_for(w)
    ybar, s2 = [], []
    for seed in range(n_seeds):
        lin, _, _ = be.render(cam, Backend.params(w, h, spp, 50, seed=1000 + seed, variant="bvh", moments=True))
        err, nz = be.noise(0.0)
        assert nz["samples"] == spp
        y = lin[..., :3].astype(np.float64) @ LUMA
        sigma = 2.0 * err.astype(np.float64) * np.sqrt(np.maximum(y, FLOOR))   # e = sigma / (2 sqrt(max(Ybar, floor)))
        ybar.append(y)
        s2.append(sigma ** 2 * spp)
    ybar, s2 = np.array(ybar), np.array(s2)
    est = s2.mean(axis=0) / spp            # estimated variance of a pixel's 16-spp mean
    emp = ybar.var(axis=0, ddof=1)         # its variance across the 32 seeds
    ratio = est.mean() / emp.mean()
    corr = np.corrcoef(est.ravel(), emp.ravel())[0, 1]
    print(f"frame-mean sigma^2: estimated {est.mean():.6g}, across seeds {emp.mean():.6g} (ratio {ratio:.4f}); per-pixel corr {corr:.4f}")
    assert abs(ratio - 1) < 0.05
    assert corr > 0.9

    # The oracle's per-path variance from 128 one-sample renders per pixel (the f64 reference, unchanged).  Its own
    # seed-to-seed spread, measured: frame means of three independent 64-path sets 0.021608 / 0.021688 / 0.021685 (0.4 %),
    # halves of one set within 0.3 %.  The bound below leaves room for that and for FP32 against f64 geometry (measured on a
    # B200: GPU / oracle 1.0018, estimated / across-seed sigma^2 0.998, per-pixel correlation 0.944).
    osc = oracle.Scene.from_arrays(scene)
    ocam, _ = oracle.default_camera(w)
    paths = np.array([osc.render(ocam, w, h, 1, 50, seed=7000 + k, threads=0)[0] @ LUMA for k in range(128)])
    o_s2 = paths.var(axis=0, ddof=1).mean()
    halves = paths[:64].var(axis=0, ddof=1).mean(), paths[64:].var(axis=0, ddof=1).mean()
    g_s2 = s2.mean()
    print(f"frame-mean per-path s^2: GPU {g_s2:.6g}, oracle {o_s2:.6g} (ratio {g_s2 / o_s2:.4f}); "
          f"oracle halves {halves[0]:.6g} / {halves[1]:.6g} (spread {abs(halves[0] / halves[1] - 1):.4f})")
    assert abs(g_s2 / o_s2 - 1) < 0.02


# ------------------------------------------------------------------------------- 5. render_to_noise
def test_render_to_noise_reaches_target_on_the_doubling_schedule(be):
    w, v = 160, "bvh"
    cam, h = cam_for(w)
    _, _, _, nz4 = single(be, cam, w, h, 4, v, seed=5)
    target = nz4["rms_err"] / 3    # about 9x the samples: 4 -> 8 -> 16 -> 32 -> 64
    lin, rgb8, n, nz = be.render_to_noise(cam, Backend.params(w, h, 4, 50, seed=5, variant=v), target, 4096)
    spp, reached_rgb8 = nz["samples"], rgb8
    assert spp >= 8 and spp % 4 == 0 and ((spp // 4) & (spp // 4 - 1)) == 0, spp   # 4 * 2^k
    assert nz["rms_err"] <= target and n == w * h * spp
    want = single(be, cam, w, h, spp, v, seed=5)
    assert np.array_equal(lin, want[0]) and np.array_equal(rgb8, want[1])
    assert {k: want[3][k] for k in ("samples", "mean_err", "rms_err", "max_err")} == {k: nz[k] for k in ("samples", "mean_err", "rms_err", "max_err")}
    assert single(be, cam, w, h, spp // 2, v, seed=5)[3]["rms_err"] > target   # it did not stop early: the previous step missed

    # max_spp too small: 4 + 4 + 4 samples (the last batch capped), RZ_OK, the target not reached
    lin, rgb8, n, nz = be.render_to_noise(cam, Backend.params(w, h, 4, 50, seed=5, variant=v), 1e-6, 12)
    assert nz["samples"] == 12 and nz["rms_err"] > 1e-6 and n == w * h * 12
    want = single(be, cam, w, h, 12, v, seed=5)
    assert np.array_equal(lin, want[0]) and np.array_equal(rgb8, want[1])
    with pytest.raises(abi.BackendError):
        be.render_to_noise(cam, Backend.params(w, h, 16, 50, seed=5, variant=v), 0.01, 8)

    # the Tracer takes the same path
    t = rayz_b200.random_bouncing(160, seed=42)
    t.samples_per_px, t.variant, t.seed = 4, v, 5
    assert t.render(noise_target=target, max_spp=4096) == w * h * spp
    assert t.noise["samples"] == spp and np.array_equal(t.img.rgb8, reached_rgb8)


# ------------------------------------------------------------------------------- 6. several devices
def _n_gpus():
    import torch
    return torch.cuda.device_count()


@pytest.mark.skipif("_n_gpus() < 2")
def test_multi_device_batches_equal_single_device_render(scene):
    import torch
    n = min(_n_gpus(), 4)
    w = 320
    cam, h = cam_for(w)
    one = Backend((0,))
    one.upload_scene(scene)
    many = Backend(tuple(range(n)))
    many.upload_scene(scene)
    for v in ("mega", "bvh"):
        want = single(one, cam, w, h, 24, v)
        assert_same(batches(many, cam, w, h, [0, 3, 8, 24], v), want)
        # page-locked host buffers: every device copies its own bands (no gather); accumulating is unchanged
        many.render(cam, Backend.params(w, h, 3, 50, seed=3, variant=v, moments=True))
        many.render(cam, Backend.params(w, h, 5, 50, seed=3, sample_offset=3, variant=v, moments=True, accumulate=True))
        pl = torch.empty((h, w, 4), dtype=torch.float32).pin_memory().numpy()
        p8 = torch.empty((h, w, 3), dtype=torch.uint8).pin_memory().numpy()
        many.render(cam, Backend.params(w, h, 16, 50, seed=3, sample_offset=8, variant=v, moments=True, accumulate=True),
                    out_linear=pl, out_rgb8=p8)
        assert np.array_equal(pl, want[0]) and np.array_equal(p8, want[1])
        assert np.array_equal(many.noise(2 / 255)[0], want[2])
    one.close()
    many.close()
