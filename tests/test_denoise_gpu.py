"""GPU tests of the denoiser (rayz_cuda_denoise): the GPU filter against the numpy f64 reference of tests/test_denoise_cpu.py
on the public readouts (render linear, noise error, guides), the exact pass-through at 0 iterations, adaptive input, no side
effects, every refusal, the quality gain against a 4096-spp frame, device-count independence and the C++ host's --denoise.

Tolerance of the reference parity: the GPU evaluates the same formulas in f32.  Each weight's exponent is rounded to a few
ulp (2^-24) of its size, and the cosine's rounding is raised to the power sigma_n = 128; through five levels of normalised
weighted means that moves a filtered value by a small multiple of 1e-4 of the values it averages (measured on one B200:
at most 6e-6 of |ref| + 1e-2 on the frames here).  The bound |gpu - ref| <= 2e-3 (|ref| + 1e-2) leaves an order of magnitude
for pixels whose neighbours are far brighter than they are (the 1e-2 term: about one 8-bit step of a dark displayed
value)."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import rayz_b200
from rayz_b200 import Backend
from rayz_b200 import _abi as abi
from test_denoise_cpu import denoise_ref, quantise_ref

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
W, SEED = 160, 3


def cam_for(w, look_from=(13, 2, 3)):
    h = int(w / rayz_b200.ASPECT_RATIO)
    return rayz_b200.Camera.init(20.0, 10.0, 0.6, look_from, (0, 0, 0), (0, 1, 0), h, w).rz, h


def params(w, h, spp, **kw):
    kw.setdefault("seed", SEED)
    kw.setdefault("variant", "bvh")
    return Backend.params(w, h, spp, 50, **kw)


@pytest.fixture(scope="module")
def scene():
    return rayz_b200.random_bouncing(W, seed=42).pool.arrays()


@pytest.fixture(scope="module")
def be(scene):
    b = Backend((0,))
    b.upload_scene(scene)
    yield b
    b.close()


def _n_gpus():
    import torch
    return torch.cuda.device_count()


def assert_matches_reference(got, lin, err, alb, nrm, **kw):
    lin_d, rgb8_d = got
    ref = denoise_ref(lin, err, alb, nrm, **kw)
    d = np.abs(lin_d[..., :3].astype(np.float64) - ref)
    assert (d <= 2e-3 * (np.abs(ref) + 1e-2)).all(), float((d / (np.abs(ref) + 1e-2)).max())
    assert (lin_d[..., 3] == 1).all()
    assert np.array_equal(rgb8_d, quantise_ref(lin_d[..., :3]))
    return float((d / (np.abs(ref) + 1e-2)).max())


# ------------------------------------------------------------------------------- 1. reference parity
@pytest.mark.parametrize("spp,kw", [(8, {}), (8, {"iterations": 3, "sigma_luminance": 1.5, "sigma_normal": 32.0, "sigma_depth": 0.5}),
                                    (8, {"iterations": 10}), (1, {})])
def test_reference_parity(be, spp, kw):
    """spp = 1: every pixel's error is +inf (n < 2), so v = +inf, w_l = 1 and the variance guard's inf path is compared."""
    cam, h = cam_for(W)
    lin, _, _ = be.render(cam, params(W, h, spp, moments=True))
    err, _ = be.noise()
    assert np.isinf(err).all() == (spp == 1)
    alb, nrm = be.guides(cam, params(W, h, 8))
    worst = assert_matches_reference(be.denoise(**kw), lin, err, alb, nrm, **kw)
    print(f"denoise parity {spp} spp {kw}: worst |gpu - ref| / (|ref| + 1e-2) = {worst:.2e}")


def test_guides_of_another_sample_range(be):
    cam, h = cam_for(W)
    lin, _, _ = be.render(cam, params(W, h, 32, moments=True))
    err, _ = be.noise()
    alb, nrm = be.guides(cam, params(W, h, 4, sample_offset=100))
    assert_matches_reference(be.denoise(), lin, err, alb, nrm)


# ------------------------------------------------------------------------------- 2. iterations = 0
def test_zero_iterations_return_the_resolved_frame(be):
    cam, h = cam_for(W)
    lin, rgb8, _ = be.render(cam, params(W, h, 8, moments=True))
    be.guides(cam, params(W, h, 2))
    lin0, rgb80 = be.denoise(iterations=0)
    assert np.array_equal(lin0.view(np.uint32), lin.view(np.uint32)) and np.array_equal(rgb80, rgb8)


# ------------------------------------------------------------------------------- 3. adaptive input
def test_adaptive_frame_uses_each_pixels_count(be):
    cam, h = cam_for(W)
    be.render(cam, params(W, h, 4, moments=True))
    target = float(np.quantile(be.noise(0.0)[0], 0.5) / 4)
    lin, _, _, _ = be.render_to_noise(cam, params(W, h, 4), target, 64, adaptive=True)
    assert len(np.unique(be.pixel_samples())) > 1
    err, _ = be.noise()
    alb, nrm = be.guides(cam, params(W, h, 8))
    assert_matches_reference(be.denoise(), lin, err, alb, nrm)


# ------------------------------------------------------------------------------- 4. no side effects
def test_denoise_leaves_the_accumulation_alone(be):
    cam, h = cam_for(W)

    def sequence(with_denoise):
        be.render(cam, params(W, h, 4, moments=True, collect_stats=True))
        be.guides(cam, params(W, h, 4))
        if with_denoise:
            s, t = be.stats(), be.timing()
            a = be.denoise()
            b = be.denoise()
            assert all(np.array_equal(x, y) for x, y in zip(a, b))   # two calls, identical bytes
            assert be.stats() == s and be.timing() == t
        lin, rgb8, _ = be.render(cam, params(W, h, 4, sample_offset=4, moments=True, accumulate=True))
        err, nz = be.noise(0.01)
        return lin, rgb8, err, nz, be.pixel_samples()

    want, got = sequence(False), sequence(True)
    for x, y in zip(got, want):
        assert np.array_equal(x, y) if isinstance(x, np.ndarray) else x == y


def test_render_device_buffers_stay(be):
    """rayz_cuda_render_device's caller may still hold its device frame: the denoiser writes buffers of its own."""
    import torch
    cam, h = cam_for(W)
    p = params(W, h, 4, moments=True)
    lin, _, _ = be.render(cam, p)
    dl, _, _ = be.render_device(cam, p)   # the same samples: the device frame holds `lin`
    be.guides(cam, params(W, h, 4))
    be.denoise()

    class Frame:
        __cuda_array_interface__ = {"shape": (lin.size,), "typestr": "<f4", "data": (dl, False), "version": 2}
    dev = torch.as_tensor(Frame(), device="cuda:0").cpu().numpy()
    assert np.array_equal(dev.reshape(lin.shape), lin)


# ------------------------------------------------------------------------------- 5. refusals
def test_refusals(be, scene):
    cam, h = cam_for(W)
    lib = be.lib
    out = np.zeros((h, W, 4), dtype=np.float32)
    out8 = np.zeros((h, W, 3), dtype=np.uint8)

    def call(b=be, **fields):
        dp = abi.RzDenoiseParams()
        dp.struct_size = C.sizeof(abi.RzDenoiseParams)
        dp.iterations = 5
        for k, v in fields.items():
            setattr(dp, k, v)
        return b.lib.rayz_cuda_denoise(b._h, C.byref(dp), out.ctypes.data, out8.ctypes.data)

    def refused(code, rc, text):
        assert rc == code, (rc, lib.rayz_cuda_last_error())
        msg = lib.rayz_cuda_last_error()
        assert msg.startswith(b"denoise:") and text in msg, msg
        assert (out == 0).all() and (out8 == 0).all()

    fresh = Backend((0,))
    fresh.upload_scene(scene)
    refused(-1, call(fresh), b"no accumulated render")
    fresh.close()

    be.render(cam, params(W, h, 4))
    be.guides(cam, params(W, h, 4))
    refused(-1, call(), b"RZ_RENDER_MOMENTS")

    be.render(cam, params(W, h, 4, moments=True))
    be.guides(cam, params(W, h, 4))
    for kw, text in (({"struct_size": 20}, b"struct_size"), ({"iterations": 11}, b"iterations"),
                     ({"sigma_luminance": -1.0}, b"sigma"), ({"sigma_normal": float("nan")}, b"sigma"),
                     ({"sigma_depth": float("inf")}, b"sigma")):
        refused(-1, call(**kw), text)
    assert call(iterations=10) == 0
    out[:] = 0
    out8[:] = 0

    cam2, _ = cam_for(W, look_from=(13, 2.5, 3))
    for gp, gcam in ((params(W, h, 4, seed=SEED + 1), cam), (params(W, h + 2, 4), cam), (params(W, h, 4), cam2)):
        be.guides(gcam, gp)
        refused(-1, call(), b"frame, camera or seed")
    be.guides(cam, params(W, h, 4))
    assert call() == 0
    out[:] = 0
    out8[:] = 0
    # a failed guides call ends the guides
    assert lib.rayz_cuda_render_guides(be._h, C.byref(cam), C.byref(params(W, h, 0)), None, None) == -1
    refused(-1, call(), b"no guide buffers")
    # a reserve of another frame ends them
    be.guides(cam, params(W, h, 4))
    be.reserve(params(W * 2, h, 4))
    be.render(cam, params(W, h, 4, moments=True))
    refused(-1, call(), b"no guide buffers")
    # a scene upload ends both the accumulation and the guides: valid guides of a moments frame, then the upload; render
    # again, and the guides of the old scene are still gone
    be.guides(cam, params(W, h, 4))
    assert call() == 0
    out[:] = 0
    out8[:] = 0
    be.upload_scene(scene)
    be.render(cam, params(W, h, 4, moments=True))
    refused(-1, call(), b"no guide buffers")
    # a shard: its rows are not image neighbours
    sp = params(W, h, 4, moments=True, shard_index=1, shard_count=3)
    be.render(cam, sp)
    be.guides(cam, sp)
    refused(-5, call(), b"shard")


def test_refusals_touch_nothing(be):
    cam, h = cam_for(W)
    be.render(cam, params(W, h, 4, moments=True, collect_stats=True))
    be.guides(cam, params(W, h, 4, seed=SEED + 1))
    before = (be.noise(0.01), be.pixel_samples(), be.stats(), be.timing())
    with pytest.raises(abi.BackendError) as e:
        be.denoise()
    assert e.value.code == -1
    after = (be.noise(0.01), be.pixel_samples(), be.stats(), be.timing())
    assert np.array_equal(before[0][0], after[0][0]) and before[0][1] == after[0][1]
    assert np.array_equal(before[1], after[1]) and before[2:] == after[2:]


# ------------------------------------------------------------------------------- 6. quality
def test_denoising_halves_the_error_of_an_8spp_frame(scene, record_property):
    """Guides of 64 camera samples under the 8-spp frame: first hits only, they cost about as much as one more sample of the
    render.  Guides of the frame's own 8 samples carry the sub-pixel texture noise of the distant checkered ground into the
    remodulated output; measured on one B200 (seed 3): denoised / noisy MSE 0.56 with them, 0.30 with 64-spp guides.  The
    own-sample ratio is recorded too and held below 0.65, so that a regression of the cheap-guide path shows."""
    w = 320
    cam, h = cam_for(w)
    b = Backend((0,))
    b.upload_scene(scene)
    ref, _, _ = b.render(cam, params(w, h, 4096, sample_offset=8))   # independent samples of the same seed
    noisy, _, _ = b.render(cam, params(w, h, 8, moments=True))
    b.guides(cam, params(w, h, 8))
    den_own, _ = b.denoise()
    b.guides(cam, params(w, h, 64))
    den, _ = b.denoise()
    b.close()
    mse = lambda x: float(((x[..., :3].astype(np.float64) - ref[..., :3]) ** 2).mean())
    ratio, ratio_own = mse(den) / mse(noisy), mse(den_own) / mse(noisy)
    record_property("denoised_over_noisy_mse", ratio)
    record_property("denoised_over_noisy_mse_own_sample_guides", ratio_own)
    print(f"320 x 180, 8 spp: noisy MSE {mse(noisy):.3e}, denoised MSE {mse(den):.3e} (64-spp guides), ratio {ratio:.3f}; "
          f"with 8-spp guides {mse(den_own):.3e}, ratio {ratio_own:.3f}")
    assert ratio <= 0.5, ratio
    assert ratio_own <= 0.65, ratio_own


# ------------------------------------------------------------------------------- 7. multi-device
@pytest.mark.skipif("_n_gpus() < 2")
def test_multi_device_equals_single_device(be, scene):
    cam, h = cam_for(W)
    many = Backend(tuple(range(min(_n_gpus(), 4))))
    many.upload_scene(scene)
    got = []
    for b in (be, many):
        b.render(cam, params(W, h, 8, moments=True))
        b.guides(cam, params(W, h, 4))
        got.append(b.denoise())
    many.close()
    for x, y in zip(*got):
        assert np.array_equal(x.view(np.uint8), y.view(np.uint8))


# ------------------------------------------------------------------------------- 8. the C++ host
def read_p3(path):
    tok = open(path).read().split()
    assert tok[0] == "P3" and tok[3] == "255"
    w, h = int(tok[1]), int(tok[2])
    return np.array(tok[4:], dtype=np.int64).reshape(h, w, 3)


def test_cpp_host_denoise_matches_backend(tmp_path):
    subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "host")], check=True)
    exe = os.path.join(ROOT, "host", "_build", "rayz_host")
    out = tmp_path / "d.ppm"
    r = subprocess.run([exe, str(W), str(tmp_path / "o.ppm"), "--spp", "4", "--seed", "42", "--render-seed", "5", "--denoise", str(out)],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    t = rayz_b200.random_bouncing(W, seed=42)
    t.samples_per_px, t.seed = 4, 5
    t.render(moments=True)
    t.render_guides()
    lin, rgb8 = t.denoise()
    assert t.denoised[1] is rgb8
    assert np.array_equal(read_p3(out), rgb8)
    assert np.array_equal(read_p3(tmp_path / "o.ppm"), t.img.rgb8)   # the normal output is the render's
    t.backend.close()
