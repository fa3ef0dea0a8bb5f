"""GPU tests of adaptive sampling: rayz_cuda_render_to_noise with RZ_RENDER_ADAPTIVE and rayz_cuda_pixel_samples.

Every path is a pure function of (seed, global pixel, sample index, bounce) and radiance is summed in integers, so a pixel that
ends an adaptive render with c samples must equal the same pixel of a uniform c-spp render of the same kernel family bit for
bit: linear, rgb8 and error."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

import rayz_b200
from rayz_b200 import Backend
from rayz_b200 import _abi as abi

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
W, SPP, MAX_SPP, OFFSET, SEED = 160, 4, 100, 5, 3
FAMILY = {"bvh": "bvh", "auto": "bvh", "mega": "mega", "mega_single": "mega_single", "wavefront": "wavefront"}


@pytest.fixture(scope="module")
def scene():
    return rayz_b200.random_bouncing(W, seed=42).pool.arrays()


@pytest.fixture(scope="module")
def be(scene):
    b = Backend((0,))
    b.upload_scene(scene)
    yield b
    b.close()


def cam_for(w):
    h = int(w / rayz_b200.ASPECT_RATIO)
    return rayz_b200.Camera.init(20.0, 10.0, 0.6, (13, 2, 3), (0, 0, 0), (0, 1, 0), h, w).rz, h


def schedule():
    """The counts a pixel can end with: SPP * 2^k, the last step capped at MAX_SPP."""
    s = [SPP]
    while s[-1] < MAX_SPP:
        s.append(s[-1] + min(s[-1], MAX_SPP - s[-1]))
    return s


@pytest.fixture(scope="module")
def target(be):
    """A per-pixel target that the sky meets at SPP and the noisiest pixels do not meet at MAX_SPP."""
    cam, h = cam_for(W)
    be.render(cam, Backend.params(W, h, SPP, 50, seed=SEED, sample_offset=OFFSET, variant="bvh", moments=True))
    err, _ = be.noise(0.0)
    return float(np.quantile(err, 0.5) / 4)


def adaptive(be, cam, h, variant, target, **kw):
    p = Backend.params(W, h, SPP, 50, seed=SEED, sample_offset=OFFSET, variant=variant, **kw)
    lin, rgb8, paths, nz = be.render_to_noise(cam, p, target, MAX_SPP, adaptive=True)
    err, _ = be.noise(target)
    return lin, rgb8, err, be.pixel_samples(), paths, nz


def uniform(be, cam, h, spp, variant, **kw):
    lin, rgb8, _ = be.render(cam, Backend.params(W, h, spp, 50, seed=SEED, sample_offset=OFFSET, variant=variant, moments=True, **kw))
    err, nz = be.noise(0.0)
    return lin, rgb8, err, nz


# ------------------------------------------------------------------------------- 1. every pixel == the uniform render of its count
@pytest.mark.parametrize("variant", ["bvh", "auto", "mega", "mega_single", "wavefront"])
def test_pixels_equal_uniform_render_of_their_count(be, target, variant):
    cam, h = cam_for(W)
    lin, rgb8, err, counts, _, _ = adaptive(be, cam, h, variant, target)
    distinct = np.unique(counts)
    assert len(distinct) >= 3, distinct
    for c in distinct:
        m = counts == c
        u = uniform(be, cam, h, int(c), FAMILY[variant])
        for got, want, name in ((lin, u[0], "linear"), (rgb8, u[1], "rgb8"), (err, u[2], "err")):
            assert np.array_equal(got[m], want[m]), f"{variant}, count {c}: {name} differs in {int((got[m] != want[m]).sum())} values"


# ------------------------------------------------------------------------------- 2. the stopping contract
def test_stopping_contract(be, target):
    cam, h = cam_for(W)
    lin, rgb8, err, counts, paths, nz = adaptive(be, cam, h, "bvh", target)
    steps = schedule()
    assert set(np.unique(counts).tolist()) <= set(steps)
    top = int(counts.max())
    assert nz["samples"] == top and nz["n_pixels"] == W * h
    assert (err[counts < top] <= target).all()
    assert nz["max_err"] <= target or nz["samples"] == MAX_SPP
    assert paths == int(counts.sum(dtype=np.uint64))
    assert counts.sum() < counts.size * top   # the sky retired early
    _, again = be.noise(target)
    assert again == nz
    # the policy itself, step by step: a pixel leaves at the first count whose error meets the target, and never comes back
    for s in steps:
        if s > top:
            break
        e = uniform(be, cam, h, s, "bvh")[2]
        assert (e[counts > s] > np.float32(target)).all(), s
        if s < MAX_SPP:
            assert (e[counts == s] <= np.float32(target)).all(), s


# ------------------------------------------------------------------------------- 3. shards
def test_shards_assemble_the_full_frame(be, target):
    cam, h = cam_for(W)
    full = adaptive(be, cam, h, "bvh", target)
    parts = [np.empty_like(x) for x in full[:4]]
    for s in range(3):
        got = adaptive(be, cam, h, "bvh", target, shard_index=s, shard_count=3, band_rows=3)
        rows = [j for j in range(h) if (j // 3) % 3 == s]
        for f, x in zip(parts, got[:4]):
            f[rows] = x
    for f, x, name in zip(parts, full[:4], ("linear", "rgb8", "err", "counts")):
        assert np.array_equal(f, x), name


# ------------------------------------------------------------------------------- 4. refusals
def _code(fn):
    with pytest.raises(abi.BackendError) as e:
        fn()
    return e.value.code


def test_refusals(be, scene, target):
    cam, h = cam_for(W)
    p = Backend.params(W, h, SPP, 50, seed=SEED, variant="bvh", moments=True)
    p.flags |= abi.RENDER_ADAPTIVE
    assert _code(lambda: be.render(cam, p)) == -1 and b"RZ_RENDER_ADAPTIVE" in be.lib.rayz_cuda_last_error()
    assert _code(lambda: be.render_device(cam, p)) == -1 and b"RZ_RENDER_ADAPTIVE" in be.lib.rayz_cuda_last_error()
    be.reserve(p)   # reserve accepts it

    # no RZ_RENDER_ACCUMULATE batch continues an adaptive frame; its sums stay as they were
    _, _, err, counts, _, nz = adaptive(be, cam, h, "bvh", target)
    top = int(counts.max())
    more = Backend.params(W, h, top, 50, seed=SEED, sample_offset=OFFSET + top, variant="bvh", moments=True, accumulate=True)
    assert _code(lambda: be.render(cam, more)) == -1
    msg = be.lib.rayz_cuda_last_error()
    assert b"RZ_RENDER_ACCUMULATE refused" in msg and b"adaptively" in msg
    err2, nz2 = be.noise(target)
    assert np.array_equal(err2, err) and nz2 == nz and np.array_equal(be.pixel_samples(), counts)

    with pytest.raises(abi.BackendError) as e:
        be.render_to_noise(cam, Backend.params(W, h, 16, 50, seed=SEED, variant="bvh"), target, 8, adaptive=True)
    assert e.value.code == -1

    # a round that fails (a traversal stack the kernel believes in overflows: RZ_ERR_INTERNAL) ends the accumulation
    be.set_tuning(debug_stack_cap=2)
    try:
        assert _code(lambda: adaptive(be, cam, h, "bvh", target)) == -7
    finally:
        be.set_tuning(debug_stack_cap=0)
    assert _code(lambda: be.noise(target)) == -1
    assert _code(lambda: be.pixel_samples()) == -1
    assert _code(lambda: Backend((0,)).pixel_samples()) == -1


# ------------------------------------------------------------------------------- 5. pixel_samples after uniform renders; the C++ host
def test_pixel_samples_of_a_uniform_frame(be):
    cam, h = cam_for(W)
    be.render(cam, Backend.params(W, h, 6, 50, seed=SEED, variant="mega"))
    c = be.pixel_samples()
    assert c.shape == (h, W) and c.dtype == np.uint32 and (c == 6).all()
    be.render(cam, Backend.params(W, h, 5, 50, seed=SEED, sample_offset=6, variant="mega", accumulate=True))
    assert (be.pixel_samples() == 11).all()
    be.render(cam, Backend.params(W, h, 7, 50, seed=SEED, variant="bvh", shard_index=1, shard_count=3, band_rows=3))
    c = be.pixel_samples()
    assert c.shape == (be.lib.rayz_cuda_shard_rows(h, 1, 3, 3), W) and (c == 7).all()


def test_cpp_host_adaptive_matches_tracer(target, tmp_path):
    subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "host")], check=True)
    exe = os.path.join(ROOT, "host", "_build", "rayz_host")
    ppm = tmp_path / "out.ppm"
    target = float(np.float32(target))   # the float both hosts pass on
    r = subprocess.run([exe, str(W), str(ppm), "--spp", str(SPP), "--seed", "42", "--noise-target", repr(target), "--max-spp", str(MAX_SPP),
                        "--adaptive"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    assert re.search(r"^Finished render \((\d+\.\d\d)s\): (\d+\.\d\d) rps and (\d+\.\d\d) us per ray$", r.stderr, re.M), r.stderr
    m = re.search(r"adaptive: (\d+) paths, mean ([\d.]+) spp, max (\d+) spp, max error ([\d.]+)", r.stderr)
    assert m, r.stderr
    t = rayz_b200.random_bouncing(W, seed=42)
    t.samples_per_px = SPP
    paths = t.render(noise_target=target, max_spp=MAX_SPP, adaptive=True)
    h = t.img.h
    want = f"P3\n{W} {h}\n255\n" + "".join(f"{a} {b} {c}\n" for a, b, c in t.img.rgb8.reshape(-1, 3).tolist())
    assert ppm.read_bytes() == want.encode()
    assert int(m.group(1)) == paths == int(t.pixel_samples.sum(dtype=np.uint64))
    assert int(m.group(3)) == t.noise["samples"] == int(t.pixel_samples.max())


# ------------------------------------------------------------------------------- 6. several devices
def _n_gpus():
    import torch
    return torch.cuda.device_count()


@pytest.mark.skipif("_n_gpus() < 2")
def test_multi_device_equals_single_device(scene, target):
    import torch
    n = min(_n_gpus(), 4)
    cam, h = cam_for(W)
    one = Backend((0,))
    one.upload_scene(scene)
    many = Backend(tuple(range(n)))
    many.upload_scene(scene)
    for v in ("bvh", "mega"):
        want = adaptive(one, cam, h, v, target)
        got = adaptive(many, cam, h, v, target)
        for x, y, name in zip(got, want, ("linear", "rgb8", "err", "counts", "paths", "summary")):
            assert np.array_equal(x, y) if isinstance(x, np.ndarray) else x == y, (v, name)
        # page-locked host buffers
        pl = torch.empty((h, W, 4), dtype=torch.float32).pin_memory().numpy()
        p8 = torch.empty((h, W, 3), dtype=torch.uint8).pin_memory().numpy()
        prm = Backend.params(W, h, SPP, 50, seed=SEED, sample_offset=OFFSET, variant=v)
        prm.flags |= abi.RENDER_ADAPTIVE
        n, nz = C.c_uint64(), abi.RzNoise()
        abi.check(many.lib.rayz_cuda_render_to_noise(many._h, C.byref(cam), C.byref(prm), target, MAX_SPP, pl.ctypes.data, p8.ctypes.data,
                                                     C.byref(n), C.byref(nz)))
        assert np.array_equal(pl, want[0]) and np.array_equal(p8, want[1]) and n.value == want[4]
        assert np.array_equal(many.pixel_samples(), want[3])
    one.close()
    many.close()
