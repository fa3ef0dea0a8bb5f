"""GPU tests of the ID mattes (rayz_cuda_render_mattes): the first-hit ids of the camera samples a render traces, ranked per
pixel by exact coverage.

Small frames, as tests/test_guides_gpu.py: against the guides' coverage (the same walk), against the f64 replay's first hits
(tests/mattes_replay.py) on the replay scenes, a synthetic scene whose pixels see hundreds of spheres each, the format, the
invariances, the state the call leaves alone, the refusals and the C++ host."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import oracle
import rayz_b200
from rayz_b200 import Backend
from rayz_b200 import _abi as abi
import mattes_replay
import replay_scenes

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
W, SEED = 160, 3
SAMPLERS = {"philox": {}, "sobol": {"sobol": True}, "sobol-rqmc": {"sobol": True, "rqmc": True, "moments": True}}


def cam_for(w, defocus=0.6):
    h = int(w / rayz_b200.ASPECT_RATIO)
    return rayz_b200.Camera.init(20.0, 10.0, defocus, (13, 2, 3), (0, 0, 0), (0, 1, 0), h, w).rz, h


@pytest.fixture(scope="module")
def scene():
    return rayz_b200.random_bouncing(W, seed=42).pool.arrays()


@pytest.fixture(scope="module")
def be(scene):
    b = Backend((0,))
    b.upload_scene(scene)
    yield b
    b.close()


def params(h, spp, w=W, **kw):
    kw.setdefault("seed", SEED)
    kw.setdefault("variant", "bvh")
    return Backend.params(w, h, spp, kw.pop("max_depth", 50), **kw)


def counts(cov, spp):
    return np.rint(cov.astype(np.float64) * spp).astype(np.int64)


def check_format(ids, cov, spp):
    """Keys strictly ascending, RZ_MATTE_EMPTY only after the last nonzero rank, coverage = float32(n / spp) bit for bit."""
    n = counts(cov, spp)
    empty = ids == abi.MATTE_EMPTY
    assert np.array_equal(empty, n == 0)
    assert (np.diff(empty.astype(np.int8), axis=-1) >= 0).all()   # once empty, empty to the end
    assert np.array_equal(cov.view(np.uint32), np.float32(n / spp).view(np.uint32))
    assert (n.sum(axis=-1) <= spp).all() and (ids[~empty] >= -1).all()
    key = (np.int64(0xffffffff) - n) * 2 ** 32 + (ids.astype(np.int64) + 2 ** 31)
    live = ~empty[..., 1:]
    assert (np.diff(key, axis=-1)[live] > 0).all()


# ------------------------------------------------------------------------------- 1. against the guides
@pytest.mark.parametrize("sampler", list(SAMPLERS))
@pytest.mark.parametrize("defocus", [0.6, 0.0])
def test_full_histogram_against_the_guides_coverage(be, sampler, defocus):
    cam, h = cam_for(W, defocus)
    p = params(h, 16, **SAMPLERS[sampler])
    ids, cov = be.mattes(cam, p, 16)
    alb, _ = be.guides(cam, p)
    check_format(ids, cov, 16)
    n = counts(cov, 16)
    assert (n.sum(axis=-1) == 16).all()
    miss = np.where(ids == abi.MATTE_MISS, n, 0).sum(axis=-1)
    assert np.array_equal(miss, 16 - np.rint(alb[..., 3].astype(np.float64) * 16).astype(np.int64))
    assert (miss > 0).any() and (miss < 16).any() and ((n > 0).sum(axis=-1) >= 3).any()


# ------------------------------------------------------------------------------- 2. against the f64 replay
def replay_cases():
    arrays1, cam1 = replay_scenes.config1(48, 27)
    arrays1g, cam1g = replay_scenes.config1(48, 27, glass_heavy=True)
    am, cams, w, h = replay_scenes.all_materials()
    return {"config1": (arrays1, cam1, 48, 27, 0.0), "config1_glass": (arrays1g, cam1g, 48, 27, 0.0),
            "outside": (am, cams["outside"], w, h, 0.0), "in_glass": (am, cams["in_glass"], w, h, 1e-3)}


@pytest.fixture(scope="module")
def cases():
    return replay_cases()


@pytest.mark.parametrize("sampler", list(SAMPLERS))
@pytest.mark.parametrize("which", ["config1", "config1_glass", "outside", "in_glass"])
def test_histograms_against_the_replay(cases, which, sampler):
    arrays, cam, w, h, t_min = cases[which]
    spp, seed = 8, 29
    b = Backend((0,))
    b.upload_scene(arrays)
    p = Backend.params(w, h, spp, 50, seed=seed, t_min=t_min, **SAMPLERS[sampler])
    ids, cov = b.mattes(cam, p, 16)
    b.close()
    check_format(ids, cov, spp)
    sc = oracle.Scene.from_arrays(arrays)
    first, proven, _ = mattes_replay.replay_first(sc, arrays, cam, w, h, 0, spp, seed, t_min, sampler)
    assert proven.mean() >= 0.95, proven.mean()
    n_ids = len(arrays["sphere_radius"])
    ref = mattes_replay.histograms(first, n_ids)
    gpu = np.zeros_like(ref)
    n = counts(cov, spp)
    for r in range(16):
        live = ids[..., r] != abi.MATTE_EMPTY
        jj, ii = np.nonzero(live)
        gpu[jj, ii, ids[jj, ii, r] + 1] += n[jj, ii, r]
    assert (gpu.sum(axis=-1) == spp).all()
    unproven = (~proven).sum(axis=-1)
    whole = unproven == 0
    assert np.array_equal(gpu[whole], ref[whole])
    # elsewhere: every proven sample is in the GPU's histogram, and at most the unproven ones moved
    proven_hist = np.zeros_like(ref)
    jj, ii, ss = np.nonzero(proven)
    np.add.at(proven_hist, (jj, ii, first[jj, ii, ss] + 1), 1)
    assert (gpu >= proven_hist).all()
    assert (np.abs(gpu - ref).sum(axis=-1) <= 2 * unproven).all()
    print(f"{which} {sampler}: {proven.mean():.4%} proven, {whole.mean():.3%} whole pixels, "
          f"{int((gpu != ref).any(axis=-1).sum())} pixels differ")


# ------------------------------------------------------------------------------- 3. many ids in one pixel
def dense_grid():
    """64 x 64 spheres of radius 0.02, 0.05 apart in the plane z = 0, seen from 50 away through a 4 x 4 frame of 3.44 degrees:
    each pixel covers about 15 x 15 of them, half of its samples hit one."""
    pool = rayz_b200.MemPool()
    m = pool.add_diffuse(pool.add_solid((0.5, 0.5, 0.5)))
    for a in range(64):
        for b in range(64):
            pool.add_sphere(((a - 31.5) * 0.05, (b - 31.5) * 0.05, 0.0), 0.02, m)
    return pool.arrays(), rayz_b200.Camera.init(3.44, 50.0, 0.0, (0, 0, 50), (0, 0, 0), (0, 1, 0), 4, 4).rz


def test_many_ids_per_pixel_lose_no_count():
    arrays, cam = dense_grid()
    spp, seed = 1024, 5
    b = Backend((0,))
    b.upload_scene(arrays)
    ids, cov = b.mattes(cam, Backend.params(4, 4, spp, 50, seed=seed), 16)
    ids1, cov1 = b.mattes(cam, Backend.params(4, 4, spp, 50, seed=seed), 1)
    b.close()
    check_format(ids, cov, spp)
    assert np.array_equal(ids1, ids[..., :1]) and np.array_equal(cov1, cov[..., :1])
    sc = oracle.Scene.from_arrays(arrays)
    first, proven, _ = mattes_replay.replay_first(sc, arrays, cam, 4, 4, 0, spp, seed)
    ref = mattes_replay.histograms(first, len(arrays["sphere_radius"]))
    distinct = (ref > 0).sum(axis=-1)
    assert distinct.min() >= 100, distinct   # hundreds of distinct ids in a pixel
    want_ids, want_n = mattes_replay.ranked(ref, 16)
    n = counts(cov, spp)
    u = (~proven).sum(axis=-1)[..., None]   # unproven samples of the pixel: the GPU may place each of them elsewhere
    assert (n.sum(axis=-1) < spp).all() and (n[..., 15] > 0).all()   # more ids than ranks: a rest is left unranked
    # every ranked count is the replay's count of that id up to the pixel's unproven samples ...
    got_ref = np.take_along_axis(ref, np.maximum(ids, -1) + 1, axis=-1)
    assert (np.abs(n - got_ref) <= u).all()
    # ... and no id left unranked has a replay count above the last rank's by more than that: the top 16 lost none
    rest = ref.copy()
    np.put_along_axis(rest, ids + 1, 0, axis=-1)
    assert (rest.max(axis=-1) <= n[..., 15] + u[..., 0]).all()
    # with every sample proven, the ranks are the replay's top 16 exactly
    whole = u[..., 0] == 0
    assert np.array_equal(ids[whole], want_ids[whole]) and np.array_equal(n[whole], want_n[whole])
    print(f"dense grid: {distinct.min()}..{distinct.max()} ids per pixel, {proven.mean():.4%} proven, {whole.sum()} whole pixels")


# ------------------------------------------------------------------------------- 4. format and prefixes
def test_fewer_ranks_are_the_first_ranks(be):
    cam, h = cam_for(W)
    p = params(h, 40)
    ids, cov = be.mattes(cam, p, 16)
    check_format(ids, cov, 40)
    for k in (1, 3, 6, 15):
        a, c = be.mattes(cam, p, k)
        assert np.array_equal(a, ids[..., :k]) and np.array_equal(c.view(np.uint32), cov[..., :k].view(np.uint32)), k
    ids1, cov1 = be.mattes(cam, params(h, 1), 4)
    check_format(ids1, cov1, 1)
    assert (ids1[..., 1:] == abi.MATTE_EMPTY).all() and (cov1[..., 0] == 1).all()


# ------------------------------------------------------------------------------- 5. invariance
@pytest.mark.parametrize("count,band", [(3, 1), (3, 4), (8, 4)])
def test_shards_assemble_the_full_frame(be, count, band):
    cam, h = cam_for(W)
    full = be.mattes(cam, params(h, 12), 6)
    parts = [np.full_like(x, -7) for x in full]
    for s in range(count):
        got = be.mattes(cam, params(h, 12, shard_index=s, shard_count=count, band_rows=band), 6)
        rows = [j for j in range(h) if (j // band) % count == s]
        assert got[0].shape[0] == len(rows)
        for f, x in zip(parts, got):
            f[rows] = x
    for f, x in zip(parts, full):
        assert np.array_equal(f.view(np.uint32), x.view(np.uint32))


def test_two_calls_are_identical_and_the_variant_does_not_matter(be):
    cam, h = cam_for(W)
    a = be.mattes(cam, params(h, 33, sample_offset=5), 7)
    for v in ("bvh", "auto", "mega", "mega_single", "wavefront"):
        b = be.mattes(cam, params(h, 33, sample_offset=5, variant=v, max_depth=1 if v == "bvh" else 7, collect_stats=v == "auto"), 7)
        for x, y in zip(a, b):
            assert np.array_equal(x.view(np.uint32), y.view(np.uint32)), v


def _n_gpus():
    import torch
    return torch.cuda.device_count()


@pytest.mark.skipif("_n_gpus() < 2")
def test_multi_device_equals_single_device(be, scene):
    cam, h = cam_for(W)
    many = Backend(tuple(range(min(_n_gpus(), 4))))
    many.upload_scene(scene)
    for kw in ({}, {"shard_index": 1, "shard_count": 3, "band_rows": 2}):
        want = be.mattes(cam, params(h, 9, **kw), 5)
        got = many.mattes(cam, params(h, 9, **kw), 5)
        for x, y in zip(got, want):
            assert np.array_equal(x.view(np.uint32), y.view(np.uint32)), kw
    many.close()


def test_config4_against_its_guides():
    """99,856 spheres (randomBouncing, grid [-158, 158)), device LBVH: the full histogram's miss count is the guides'."""
    t = rayz_b200.random_bouncing(320, seed=42, grid_lo=-158, grid_hi=158)
    t.samples_per_px, t.seed = 16, 7
    ids, cov = t.render_mattes(16)
    alb, _ = t.render_guides()
    assert t.matte_ids is ids and t.matte_coverage is cov
    check_format(ids, cov, 16)
    n = counts(cov, 16)
    assert (n.sum(axis=-1) == 16).all()
    miss = np.where(ids == abi.MATTE_MISS, n, 0).sum(axis=-1)
    assert np.array_equal(miss, 16 - np.rint(alb[..., 3].astype(np.float64) * 16).astype(np.int64))
    assert len(np.unique(ids[ids >= 0])) > 1000
    t.backend.close()


# ------------------------------------------------------------------------------- 6. no side effects
def test_mattes_leave_the_accumulated_frame_and_the_guides_alone(be):
    cam, h = cam_for(W)

    def sequence(with_mattes):
        be.render(cam, params(h, 4, moments=True))
        be.guides(cam, params(h, 4))
        if with_mattes:
            be.mattes(cam, params(h, 7, seed=SEED + 1, sample_offset=2), 9)
        lin, rgb8, _ = be.render(cam, params(h, 4, sample_offset=4, moments=True, accumulate=True))
        err, nz = be.noise(0.01)
        dl, d8 = be.denoise()
        return lin, rgb8, err, nz, be.pixel_samples(), dl, d8

    want, got = sequence(False), sequence(True)
    for x, y in zip(got, want):
        assert np.array_equal(x, y) if isinstance(x, np.ndarray) else x == y


def test_mattes_leave_an_adaptive_frame_stats_and_timing_alone(be):
    cam, h = cam_for(W)
    be.render(cam, params(h, 4, moments=True, collect_stats=True))
    target = float(np.quantile(be.noise(0.0)[0], 0.5) / 4)
    be.render_to_noise(cam, params(h, 4, collect_stats=True), target, 64, adaptive=True)
    counts_, (err, nz) = be.pixel_samples(), be.noise(target)
    s, t = be.stats(), be.timing()
    assert len(np.unique(counts_)) > 1
    be.mattes(cam, params(h, 4, collect_stats=True), 6)
    err2, nz2 = be.noise(target)
    assert np.array_equal(be.pixel_samples(), counts_) and np.array_equal(err2, err) and nz2 == nz
    assert be.stats() == s and be.timing() == t


# ------------------------------------------------------------------------------- 7. refusals and faults
def test_refusals(be):
    cam, h = cam_for(W)
    lib = be.lib
    ids = np.full((h, W, 16), 77, dtype=np.int32)
    cov = np.full((h, W, 16), 0.5, dtype=np.float32)

    def call(b, p, c=cam, ranks=6):
        return lib.rayz_cuda_render_mattes(b._h if b is not None else None, C.byref(c) if c is not None else None,
                                           C.byref(p) if p is not None else None, ranks, ids.ctypes.data, cov.ctypes.data)

    def refused(code, rc, text):
        assert rc == code, (rc, lib.rayz_cuda_last_error())
        msg = lib.rayz_cuda_last_error()
        assert msg.startswith(b"mattes:") and text in msg, msg

    refused(-1, call(None, params(h, 4)), b"NULL")
    refused(-1, call(be, None), b"NULL")
    refused(-1, call(be, params(h, 4), None), b"NULL")
    refused(-1, call(be, params(h, 4), ranks=0), b"ranks")
    refused(-1, call(be, params(h, 4), ranks=17), b"ranks")
    refused(-1, call(be, params(h, 1025)), b"RZ_MATTE_MAX_SPP")
    refused(-1, call(be, params(h, 1, accumulate=True)), b"RZ_RENDER_ACCUMULATE")
    for flag, name in ((abi.RENDER_ADAPTIVE, b"RZ_RENDER_ADAPTIVE"), (abi.RENDER_ADAPTIVE_POOLED, b"RZ_RENDER_ADAPTIVE_POOLED"),
                       (abi.RENDER_PASSES, b"RZ_RENDER_PASSES")):
        p = params(h, 1)
        p.flags |= flag
        refused(-1, call(be, p), name)
    fresh = Backend((0,))
    refused(-6, call(fresh, params(h, 4)), b"rayz_cuda_upload_scene")
    fresh.close()
    refused(-1, call(be, params(h, 0)), b"spp")
    bad = params(h, 1)
    bad.variant = 9
    refused(-1, call(be, bad), b"unknown variant")
    refused(-1, call(be, params(h, 1, shard_index=3, shard_count=3)), b"shard_index")
    assert (ids == 77).all() and (cov == 0.5).all()

    # a traversal stack the kernel believes holds one entry overflows: RZ_ERR_INTERNAL, and the context stays usable
    be.set_tuning(debug_stack_cap=1)
    try:
        refused(-7, call(be, params(h, 2)), b"traversal-stack overflow")
    finally:
        be.set_tuning(debug_stack_cap=0)
    assert (ids == 77).all() and (cov == 0.5).all()
    a, c = be.mattes(cam, params(h, 2), 2)
    check_format(a, c, 2)
    lin, _, _ = be.render(cam, params(h, 2))
    assert np.isfinite(lin).all()


# ------------------------------------------------------------------------------- 8. the C++ host
def read_pfm(path):
    raw = open(path, "rb").read()
    tag, dims, scale, body = raw.split(b"\n", 3)
    w, h = (int(x) for x in dims.split())
    assert float(scale) == -1.0
    ch = {b"PF": 3, b"Pf": 1}[tag]
    return np.frombuffer(body, dtype="<f4").reshape(h, w, ch)[::-1]


def test_cpp_host_mattes_match_backend(tmp_path):
    subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "host")], check=True)
    exe = os.path.join(ROOT, "host", "_build", "rayz_host")
    prefix = str(tmp_path / "m")
    r = subprocess.run([exe, str(W), str(tmp_path / "o.ppm"), "--spp", "12", "--seed", "42", "--render-seed", "5", "--mattes", prefix],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    t = rayz_b200.random_bouncing(W, seed=42)
    t.samples_per_px, t.seed = 12, 5
    ids, cov = t.render_mattes()
    assert ids.shape[-1] == 6
    for k in range(6):
        got = read_pfm(f"{prefix}_rank{k}.pfm")
        assert np.array_equal(got[..., 0], ids[..., k].astype(np.float32))
        assert np.array_equal(got[..., 1], cov[..., k]) and (got[..., 2] == 0).all()
    t.backend.close()
    r = subprocess.run([exe, "16", str(tmp_path / "o2.ppm"), "--spp", "1025", "--mattes", prefix], capture_output=True, text=True,
                       timeout=300)
    assert r.returncode != 0 and "--mattes" in r.stderr
