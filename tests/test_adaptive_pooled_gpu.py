"""GPU tests of pooled adaptive stopping (RZ_RENDER_ADAPTIVE_POOLED with RZ_RENDER_ADAPTIVE in rayz_cuda_render_to_noise).

A pixel stops on e*, its iid error pooled with its row segment's (include/rayz_cuda.h).  The guarantees of plain adaptive
sampling hold as written (exact pixels, the contract on the estimate, shard and device invariance); what the flag adds is a
frame whose MEASURED error meets the per-pixel target, which the honesty test checks against a high-spp reference."""
import os
import re
import subprocess

import numpy as np
import pytest

import rayz_b200
from rayz_b200 import Backend
from rayz_b200 import _abi as abi

pytestmark = pytest.mark.gpu
SEED = 7
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SAMPLERS = {"philox": {}, "sobol": {"sobol": True}, "rqmc": {"sobol": True, "rqmc": True}}
NU0 = float(re.search(r"NU0 = (\d+)", open(os.path.join(ROOT, "include", "rayz_cuda.h")).read()).group(1))


@pytest.fixture(scope="module")
def scene():
    return rayz_b200.random_bouncing(400, seed=42).pool.arrays()


@pytest.fixture(scope="module")
def be(scene):
    b = Backend((0,))
    b.upload_scene(scene)
    yield b
    b.close()


def cam_for(w):
    h = int(w / rayz_b200.ASPECT_RATIO)
    return rayz_b200.Camera.init(20.0, 10.0, 0.6, (13, 2, 3), (0, 0, 0), (0, 1, 0), h, w).rz, h


def params(w, h, spp, sampler="philox", **kw):
    kw.setdefault("seed", SEED)
    kw.setdefault("variant", "bvh")
    return Backend.params(w, h, spp, kw.pop("max_depth", 50), **kw, **SAMPLERS[sampler])


def pooled_run(b, cam, p, target, max_spp):
    lin, rgb8, paths, nz = b.render_to_noise(cam, p, target, max_spp, adaptive=True, pooled=True)
    return lin, rgb8, paths, nz


def restate(err, counts, width, nu0=NU0):
    """e* from a plain frame's out_err and counts (numpy f64): u = n e^2, U_S over the segment's pixels with n >= 2.  Under
    RQMC out_err is e sqrt(G) with one G per segment, so the same arithmetic gives e* sqrt(G)."""
    n = counts.astype(np.float64)
    e = err.astype(np.float64)
    u = np.where(n >= 2, n * e * e, 0.0)
    d = np.where(n >= 2, n - 1, 0.0)
    rows = err.shape[0]
    nseg = -(-width // 64)
    seg = (np.arange(rows)[:, None] * nseg + np.arange(width)[None, :] // 64)
    num = np.bincount(seg.ravel(), (d * u).ravel(), rows * nseg)
    den = np.bincount(seg.ravel(), d.ravel(), rows * nseg)
    U = np.where(den > 0, num / np.where(den > 0, den, 1), 0.0)[seg]
    with np.errstate(divide="ignore", invalid="ignore"):
        return np.where(n >= 2, np.sqrt((nu0 * U + (n - 1) * u) / (nu0 + n - 1) / n), np.inf)


# ------------------------------------------------------------------------------- 1. refusals
def test_refusals_leave_the_accumulated_frame_untouched(be):
    w = 160
    cam, h = cam_for(w)
    lin, rgb8, _, _ = pooled_run(be, cam, params(w, h, 4), 4 / 255, 16)
    err, nz = be.noise()
    counts = be.pixel_samples()

    def refused(call, rule):
        with pytest.raises(abi.BackendError) as e:
            call()
        assert e.value.code == -1 and rule in str(e.value), str(e.value)
        err2, nz2 = be.noise()                                 # the accumulated frame is still there, as it was
        assert nz2 == nz and np.array_equal(err2, err) and np.array_equal(be.pixel_samples(), counts)

    pooled = lambda **kw: _with(params(w, h, 4, moments=True, **kw), abi.RENDER_ADAPTIVE_POOLED)
    refused(lambda: be.render_to_noise(cam, params(w, h, 4), 4 / 255, 16, pooled=True), "RZ_RENDER_ADAPTIVE_POOLED requires RZ_RENDER_ADAPTIVE")
    refused(lambda: be.render(cam, pooled()), "RZ_RENDER_ADAPTIVE_POOLED")
    refused(lambda: be.render(cam, _with(pooled(), abi.RENDER_ADAPTIVE)), "RZ_RENDER_ADAPTIVE_POOLED")
    refused(lambda: be.render_device(cam, pooled()), "RZ_RENDER_ADAPTIVE_POOLED")
    refused(lambda: be.guides(cam, pooled()), "RZ_RENDER_ADAPTIVE_POOLED")
    refused(lambda: be.guides(cam, _with(pooled(), abi.RENDER_ADAPTIVE)), "RZ_RENDER_ADAPTIVE_POOLED")
    refused(lambda: be.reserve(pooled()), "RZ_RENDER_ADAPTIVE_POOLED requires RZ_RENDER_ADAPTIVE")
    # an accumulate batch after the adaptive call: refused as before
    refused(lambda: be.render(cam, params(w, h, 4, sample_offset=16, accumulate=True, moments=True)), "rendered adaptively")
    be.reserve(_with(pooled(), abi.RENDER_ADAPTIVE))           # with ADAPTIVE the reserve takes it


def _with(p, flags):
    q = abi.RzRenderParams.from_buffer_copy(p)
    q.flags |= flags
    return q


# ------------------------------------------------------------------------------- 2. exact pixels
@pytest.mark.parametrize("variant", ["bvh", "mega"])
@pytest.mark.parametrize("sampler", list(SAMPLERS))
def test_pooled_pixels_equal_uniform_renders_of_their_count(be, variant, sampler):
    w, spp, max_spp = 160, 4, 64
    cam, h = cam_for(w)
    be.render(cam, params(w, h, spp, sampler, variant=variant, moments=True))
    target = float(np.quantile(be.noise()[0], 0.5) / 3)
    lin, rgb8, _, _ = pooled_run(be, cam, params(w, h, spp, sampler, variant=variant), target, max_spp)
    counts = be.pixel_samples()
    distinct = np.unique(counts)
    assert len(distinct) >= 3, distinct
    for c in distinct:
        m = counts == c
        ul, u8, _ = be.render(cam, params(w, h, int(c), sampler, variant=variant, moments=True))
        assert np.array_equal(lin[m], ul[m]) and np.array_equal(rgb8[m], u8[m]), (variant, sampler, c)


# ------------------------------------------------------------------------------- 3. the estimator on the device
@pytest.mark.parametrize("sampler", list(SAMPLERS))
def test_one_round_error_equals_numpy_restatement(be, sampler):
    w, spp = 200, 8                                        # segments of 64, 64, 64 and a short 8
    cam, h = cam_for(w)
    be.render(cam, params(w, h, spp, sampler, moments=True))
    plain, _ = be.noise()
    target = float(np.median(plain))
    pooled_run(be, cam, params(w, h, spp, sampler), target, spp)   # max_spp == spp: one round, no list
    err, nz = be.noise(target)
    assert (be.pixel_samples() == spp).all() and nz["samples"] == spp
    want = restate(plain, np.full(plain.shape, spp), w)
    np.testing.assert_allclose(err, want, rtol=2e-6, atol=1e-9)
    assert not np.allclose(err, plain, rtol=1e-3)          # the prior moves the errors
    assert nz["n_above"] == int((err.astype(np.float64) > np.float32(target)).sum())


# ------------------------------------------------------------------------------- 4. contract
@pytest.mark.parametrize("sampler", list(SAMPLERS))
def test_contract_on_the_estimate(be, sampler):
    w, max_spp = 240, 256
    cam, h = cam_for(w)
    target = 4 / 255
    _, _, paths, nz = pooled_run(be, cam, params(w, h, 4, sampler), target, max_spp)
    err, nz2 = be.noise(target)
    counts = be.pixel_samples()
    assert nz2 == nz
    assert nz["max_err"] <= target or nz["samples"] == max_spp
    capped = counts == max_spp
    assert (err[~capped] <= np.float32(target)).all()      # a stopped pixel keeps the prior its test read
    assert nz["n_above"] == int((err.astype(np.float64) > np.float32(target)).sum())
    assert int(counts.astype(np.int64).sum()) == paths and nz["samples"] == counts.max()
    assert nz["max_err"] == pytest.approx(float(err.max()), rel=0) and nz["n_pixels"] == w * h


# ------------------------------------------------------------------------------- 5. invariance
def test_shards_assemble_the_full_frame(be):
    w, count, band = 160, 3, 3
    cam, h = cam_for(w)
    target = 4 / 255
    full, full8, _, _ = pooled_run(be, cam, params(w, h, 4, band_rows=band), target, 128)
    full_err, _ = be.noise(target)
    full_n = be.pixel_samples()
    rows = np.arange(h)
    for s in range(count):
        lin, rgb8, _, _ = pooled_run(be, cam, params(w, h, 4, shard_index=s, shard_count=count, band_rows=band), target, 128)
        err, _ = be.noise(target)
        mine = rows[(rows // band) % count == s]
        assert np.array_equal(be.pixel_samples(), full_n[mine]) and np.array_equal(lin, full[mine])
        assert np.array_equal(rgb8, full8[mine]) and np.array_equal(err, full_err[mine]), s


def _n_gpus():
    import torch
    return torch.cuda.device_count()


@pytest.mark.skipif("_n_gpus() < 2")
def test_multi_device_equals_single_device(be, scene):
    w = 320
    cam, h = cam_for(w)
    many = Backend((0, 1))
    try:
        many.upload_scene(scene)
        for s in SAMPLERS:
            a, a8, _, _ = pooled_run(be, cam, params(w, h, 4, s), 4 / 255, 128)
            ae, an = be.noise()[0], be.pixel_samples()
            b, b8, _, _ = pooled_run(many, cam, params(w, h, 4, s), 4 / 255, 128)
            assert np.array_equal(a, b) and np.array_equal(a8, b8), s
            assert np.array_equal(ae, many.noise()[0]) and np.array_equal(an, many.pixel_samples()), s
    finally:
        many.close()


# ------------------------------------------------------------------------------- 6, 7. honesty and cost
HONEST_W = 320
luma = lambda x: 0.2126 * x[..., 0] + 0.7152 * x[..., 1] + 0.0722 * x[..., 2]
disp = lambda x: np.sqrt(np.maximum(luma(x), 1e-4))


@pytest.fixture(scope="module")
def honest():
    """Config 2 and penultimate_scene at 320 x 180, each with an 8192-spp Philox reference of two 4096-spp halves."""
    out = {}
    for name in ("config2", "penultimate"):
        t = rayz_b200.random_bouncing(HONEST_W, seed=42) if name == "config2" else rayz_b200.penultimate_scene(HONEST_W)
        h = int(HONEST_W / rayz_b200.ASPECT_RATIO)
        b = Backend((0,))
        b.upload_scene(t.pool.arrays())
        cam = t.camera.rz
        ra, _, _ = b.render(cam, Backend.params(HONEST_W, h, 4096, 50, seed=1001, variant="bvh"), want_rgb8=False)
        rc, _, _ = b.render(cam, Backend.params(HONEST_W, h, 4096, 50, seed=1002, variant="bvh"), want_rgb8=False)
        ra, rc = ra[..., :3].astype(np.float64), rc[..., :3].astype(np.float64)
        out[name] = (b, cam, h, disp((ra + rc) / 2), (disp(ra) - disp(rc)) ** 2 / 4)
    yield out
    for v in out.values():
        v[0].close()


def measured_rms(S, lin, mask):
    """rms displayed error over `mask` against the reference, the reference's own noise removed."""
    _, _, _, ref, ref_noise = S
    d2 = (disp(lin[..., :3].astype(np.float64)) - ref) ** 2 - ref_noise
    return float(np.sqrt(max(d2[mask].mean(), 0.0)))


@pytest.mark.parametrize("name", ["config2", "penultimate"])
@pytest.mark.parametrize("sampler", list(SAMPLERS))
def test_pooled_stopping_is_honest_and_cheaper_than_uniform(honest, name, sampler):
    S = honest[name]
    b, cam, h = S[0], S[1], S[2]
    target, max_spp = 2 / 255, 4096
    p = Backend.params(HONEST_W, h, 4, 50, seed=SEED, variant="bvh", **SAMPLERS[sampler])
    lin, _, paths, nz = pooled_run(b, cam, p, target, max_spp)
    counts = b.pixel_samples()
    live = counts < max_spp
    ratio = measured_rms(S, lin, live) / target
    groups = {int(c): measured_rms(S, lin, counts == c) / target for c in np.unique(counts[live]) if (counts == c).sum() >= 2000}
    plin, _, ppaths, _ = b.render_to_noise(cam, p, target, max_spp, adaptive=True)
    pcounts = b.pixel_samples()
    plain = measured_rms(S, plin, pcounts < max_spp) / target
    # uniform doubling until the frame's max estimate meets the target, the bound adaptive sampling gives
    q = Backend.params(HONEST_W, h, 4, 50, seed=SEED, variant="bvh", moments=True, **SAMPLERS[sampler])
    b.render(cam, q, want_linear=False, want_rgb8=False)
    n = 4
    while b.noise()[1]["max_err"] > target and n < max_spp:
        q = Backend.params(HONEST_W, h, min(n, max_spp - n), 50, seed=SEED, sample_offset=n, variant="bvh", accumulate=True, moments=True,
                           **SAMPLERS[sampler])
        b.render(cam, q, want_linear=False, want_rgb8=False)
        n += q.spp
    uniform_paths = n * HONEST_W * h
    print(f"{name} {sampler}: pooled measured/target {ratio:.3f} ({paths / 1e6:.1f} M paths, {(~live).sum()} capped), "
          f"groups {', '.join(f'{c}: {r:.2f}' for c, r in groups.items())}; plain adaptive {plain:.3f} ({ppaths / 1e6:.1f} M); "
          f"uniform to max {n} spp ({uniform_paths / 1e6:.1f} M)")
    assert ratio <= 1.1
    assert all(r <= 1.3 for r in groups.values()), groups
    assert plain > ratio
    assert paths < uniform_paths


# ------------------------------------------------------------------------------- 8. denoiser
def test_denoiser_accepts_a_pooled_frame(be):
    w = 160
    cam, h = cam_for(w)
    p = params(w, h, 4)
    lin, rgb8, _, _ = pooled_run(be, cam, p, 4 / 255, 64)
    be.guides(cam, p)
    same, same8 = be.denoise(iterations=0)
    assert np.array_equal(same, lin) and np.array_equal(same8, rgb8)
    den, _ = be.denoise()
    assert np.isfinite(den).all() and not np.array_equal(den, lin)


# ------------------------------------------------------------------------------- 9. C++ host
def test_cpp_host_pooled_equals_the_tracer(tmp_path):
    subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "host")], check=True)
    exe = os.path.join(ROOT, "host", "_build", "rayz_host")
    w, ppm = 96, tmp_path / "out.ppm"
    r = subprocess.run([exe, str(w), str(ppm), "--spp", "4", "--seed", "42", "--noise-target", "0.02", "--max-spp", "64", "--adaptive",
                        "--pooled"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    assert re.search(r"^Finished render \(", r.stderr, re.M) and "adaptive:" in r.stderr
    h = int(w / rayz_b200.ASPECT_RATIO)
    lines = ppm.read_text().split("\n")
    assert lines[:3] == ["P3", f"{w} {h}", "255"] and len(lines) == 3 + w * h + 1
    t = rayz_b200.random_bouncing(w, seed=42)
    t.samples_per_px = 4
    t.render(noise_target=0.02, max_spp=64, adaptive=True, pooled=True)
    assert lines[3:-1] == [" ".join(str(int(x)) for x in px) for px in t.img.rgb8.reshape(-1, 3)]
    plain = rayz_b200.random_bouncing(w, seed=42)
    plain.samples_per_px = 4
    plain.render(noise_target=0.02, max_spp=64, adaptive=True)
    assert not np.array_equal(plain.pixel_samples, t.pixel_samples)   # the flag reached the library
    r = subprocess.run([exe, str(w), str(ppm), "--spp", "4", "--noise-target", "0.02", "--pooled"], capture_output=True, text=True, timeout=300)
    assert r.returncode != 0 and "RZ_RENDER_ADAPTIVE_POOLED requires RZ_RENDER_ADAPTIVE" in r.stderr
